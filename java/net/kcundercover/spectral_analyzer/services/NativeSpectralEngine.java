package net.kcundercover.spectral_analyzer.services;

import java.lang.foreign.Arena;
import java.lang.foreign.FunctionDescriptor;
import java.lang.foreign.Linker;
import java.lang.foreign.MemoryLayout;
import java.lang.foreign.MemorySegment;
import java.lang.foreign.StructLayout;
import java.lang.foreign.SymbolLookup;
import java.lang.foreign.ValueLayout;
import java.lang.invoke.MethodHandle;
import java.nio.MappedByteBuffer;

import static java.lang.foreign.ValueLayout.ADDRESS;
import static java.lang.foreign.ValueLayout.JAVA_DOUBLE;
import static java.lang.foreign.ValueLayout.JAVA_INT;
import static java.lang.foreign.ValueLayout.JAVA_LONG;

/**
 * Panama (java.lang.foreign) binding of libsa_engine.so -- the reference-side stub a maintainer adds.
 *
 * NOT compiled in this repository (no JVM in the build image; Java 21 needs --enable-preview for
 * java.lang.foreign, final in 22).  It binds exactly the symbols declared in include/sa_engine.h and
 * is mirrored 1:1 by spectral_analyzer_b200/_capi.py, which IS exercised by the tests.
 *
 * No JNI glue and no CPU fallback: if the library or a B200 is missing, construction throws.
 */
public final class NativeSpectralEngine implements AutoCloseable {
    private static final Linker LINKER = Linker.nativeLinker();
    private static final SymbolLookup LIB = SymbolLookup.libraryLookup(
            System.getProperty("sa.engine.lib", "libsa_engine.so"), Arena.global());

    private static MethodHandle fn(String name, FunctionDescriptor fd) {
        return LINKER.downcallHandle(LIB.find(name).orElseThrow(() -> new UnsatisfiedLinkError(name)), fd);
    }

    // int32 sa_engine_create(int32 device, sa_engine** out)
    private static final MethodHandle CREATE = fn("sa_engine_create", FunctionDescriptor.of(JAVA_INT, JAVA_INT, ADDRESS));
    private static final MethodHandle DESTROY = fn("sa_engine_destroy", FunctionDescriptor.ofVoid(ADDRESS));
    private static final MethodHandle LAST_ERROR = fn("sa_last_error", FunctionDescriptor.of(ADDRESS));
    private static final MethodHandle PARSE_DT = fn("sa_parse_datatype", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle REGISTER = fn("sa_register_host", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT));
    private static final MethodHandle UNREGISTER = fn("sa_unregister_host", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));
    private static final MethodHandle PARAMS_INIT = fn("sa_spectrogram_params_init", FunctionDescriptor.ofVoid(ADDRESS));
    // int32 sa_spectrogram(engine, iq, iq_bytes, params, out, out_bytes)
    private static final MethodHandle SPECTROGRAM = fn("sa_spectrogram",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, JAVA_LONG));
    // int32 sa_compute_magnitudes(engine, buffer, capacity, start_byte, nfft, dtype, big_endian, out)
    private static final MethodHandle MAGNITUDES = fn("sa_compute_magnitudes",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, JAVA_INT, JAVA_INT, JAVA_INT, ADDRESS));
    // int32 sa_downconvert(engine, iq, iq_bytes, dtype, be, start, count, freq_off, down, fast, re, im, out_len)
    private static final MethodHandle DOWNCONVERT = fn("sa_downconvert",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT, JAVA_LONG, JAVA_LONG,
                    JAVA_DOUBLE, JAVA_INT, JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    // int32 sa_psd_welch(engine, re, im, n, fs, nfft, hop, window, out_freq, out_db)
    private static final MethodHandle PSD_WELCH = fn("sa_psd_welch",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_DOUBLE, JAVA_INT, JAVA_LONG,
                    JAVA_INT, ADDRESS, ADDRESS));

    // int32 sa_spectrogram_file(engine, path, data_offset, data_bytes, params, out, out_bytes)
    private static final MethodHandle SPECTROGRAM_FILE = fn("sa_spectrogram_file",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_LONG, ADDRESS, ADDRESS, JAVA_LONG));
    // uint64 sa_downconvert_length(engine, count, down, fast)
    private static final MethodHandle DOWNCONVERT_LENGTH = fn("sa_downconvert_length",
            FunctionDescriptor.of(JAVA_LONG, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT));
    // int32 sa_downconvert_psd_batch(engine, iq, iq_bytes, dtype, be, fs, anns, n_ann, psd_nfft, psd_hop, psd_window,
    //                                out_iq, iq_offsets, out_psd_db)
    private static final MethodHandle BATCH = fn("sa_downconvert_psd_batch",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, JAVA_INT, JAVA_DOUBLE, ADDRESS, JAVA_INT,
                    JAVA_INT, JAVA_LONG, JAVA_INT, ADDRESS, ADDRESS, ADDRESS));
    private static final MethodHandle CONFIG_INIT = fn("sa_analysis_config_init", FunctionDescriptor.ofVoid(ADDRESS));
    // int32 sa_set_analysis_config(engine, config)
    private static final MethodHandle SET_CONFIG = fn("sa_set_analysis_config", FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS));

    // int32 sa_render_canvas(engine, iq, iq_bytes, params, canvas_w, canvas_h, frames_per_column, reduce, out_rgba)
    private static final MethodHandle RENDER_CANVAS = fn("sa_render_canvas",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, JAVA_INT, JAVA_INT, JAVA_LONG, JAVA_INT, ADDRESS));
    // int32 sa_spectrum_trace(engine, iq, iq_bytes, params, frames_per_row, out_mean, out_max, out_min, out_bytes)
    private static final MethodHandle SPECTRUM_TRACE = fn("sa_spectrum_trace",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, JAVA_LONG, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG));
    // int32 sa_spectrum_persistence(engine, iq, iq_bytes, params*, n_levels, min_db, max_db, out_counts, out_bytes)
    private static final MethodHandle SPECTRUM_PERSISTENCE = fn("sa_spectrum_persistence",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, JAVA_LONG, ADDRESS, JAVA_INT, JAVA_DOUBLE, JAVA_DOUBLE, ADDRESS,
                                  JAVA_LONG));
    // int32 sa_iq_pack(engine, re, im, n, format, out)
    private static final MethodHandle IQ_PACK = fn("sa_iq_pack",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_INT, ADDRESS));
    // int32 sa_analysis_series(engine, re, im, n, fs, alpha_mag, alpha_freq, center_freq, out_mag_db, out_freq)
    private static final MethodHandle ANALYSIS_SERIES = fn("sa_analysis_series",
            FunctionDescriptor.of(JAVA_INT, ADDRESS, ADDRESS, ADDRESS, JAVA_LONG, JAVA_DOUBLE, JAVA_DOUBLE, JAVA_DOUBLE,
                    JAVA_DOUBLE, ADDRESS, ADDRESS));

    /** struct sa_spectrogram_params (include/sa_engine.h), natural alignment, 96 bytes. */
    static final StructLayout PARAMS = MemoryLayout.structLayout(
            JAVA_INT.withName("struct_size"), JAVA_INT.withName("dtype"), JAVA_INT.withName("big_endian"),
            JAVA_INT.withName("window"), JAVA_INT.withName("nfft"), JAVA_INT.withName("db_mode"),
            JAVA_INT.withName("out_kind"), JAVA_INT.withName("precision"), JAVA_LONG.withName("start_sample"),
            JAVA_LONG.withName("hop"), JAVA_LONG.withName("n_frames"), JAVA_DOUBLE.withName("eof_fill_db"),
            JAVA_INT.withName("colormap"), JAVA_INT.withName("strict_reference"), JAVA_DOUBLE.withName("sample_rate"),
            JAVA_DOUBLE.withName("min_db"), JAVA_DOUBLE.withName("max_db"));

    /** struct sa_annotation (include/sa_engine.h): one row of the batch loop AnnotationController.java:321-360. */
    static final StructLayout ANNOTATION = MemoryLayout.structLayout(
            JAVA_LONG.withName("start_sample"), JAVA_LONG.withName("count"), JAVA_DOUBLE.withName("freq_off"),
            JAVA_INT.withName("down"), JAVA_INT.withName("fast"));

    /** struct sa_analysis_config (include/sa_engine.h): what JDSP decides inside downConvert / calculatePsdWelch. */
    static final StructLayout CONFIG = MemoryLayout.structLayout(
            JAVA_INT.withName("struct_size"), JAVA_INT.withName("n_taps"), ADDRESS.withName("taps"),
            JAVA_INT.withName("delay_mode"), JAVA_INT.withName("length_mode"), JAVA_INT.withName("psd_scaling"),
            JAVA_INT.withName("psd_detrend"), JAVA_INT.withName("psd_precision"), JAVA_INT.withName("strict_reference"));

    private final MemorySegment engine;

    public NativeSpectralEngine(int device) {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment out = a.allocate(ADDRESS);
            check((int) CREATE.invoke(device, out));
            engine = out.get(ADDRESS, 0);
        } catch (RuntimeException e) {
            throw e;
        } catch (Throwable t) {
            throw new IllegalStateException(t);
        }
    }

    private static void check(int rc) throws Throwable {
        if (rc == 0) return;
        String msg = ((MemorySegment) LAST_ERROR.invoke()).reinterpret(512).getString(0);
        switch (rc) {
            case 1: throw new IllegalArgumentException(msg);          // MathIllegalArgumentException analogue
            case 3: throw new IndexOutOfBoundsException(msg);         // absolute get past the buffer limit
            default: throw new IllegalStateException("sa_engine " + rc + ": " + msg);
        }
    }

    /**
     * Page-locks an ANONYMOUS native segment (Arena-allocated staging or output memory) so that it is the DMA source /
     * target itself.  Do not call it with the MappedByteBuffer of SigMfHelper.load (SigMfHelper.java:78-84):
     * cudaHostRegister refuses file-backed mappings (measured on the B200 hosts: "invalid argument") and this throws.
     * The mapped buffer needs no registration: the engine stages it through its own pinned ring with parallel copies,
     * and {@link #spectrogramFromFile} reads the data file into that ring directly.
     */
    public void register(MemorySegment anonymousSegment) throws Throwable {
        check((int) REGISTER.invoke(engine, anonymousSegment, anonymousSegment.byteSize(), 0));
    }

    /**
     * The JDSP profile of this engine (sa_set_analysis_config): taps (null = built-in design), delay mode
     * (0 causal, 1 same, 2 valid), length mode (0 floor, 1 ceil), PSD scaling (0 density, 1 spectrum), detrend
     * (0 none, 1 constant), PSD precision (1 FP32, 2 FP64), strict reference decode.
     */
    public void setAnalysisConfig(double[] taps, int delayMode, int lengthMode, int psdScaling, int psdDetrend,
                                  int psdPrecision, boolean strictReference) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment c = a.allocate(CONFIG);
            CONFIG_INIT.invoke(c);
            if (taps != null) {
                c.set(ADDRESS, CONFIG.byteOffset(MemoryLayout.PathElement.groupElement("taps")), a.allocateFrom(JAVA_DOUBLE, taps));
                c.set(JAVA_INT, CONFIG.byteOffset(MemoryLayout.PathElement.groupElement("n_taps")), taps.length);
            }
            c.set(JAVA_INT, CONFIG.byteOffset(MemoryLayout.PathElement.groupElement("delay_mode")), delayMode);
            c.set(JAVA_INT, CONFIG.byteOffset(MemoryLayout.PathElement.groupElement("length_mode")), lengthMode);
            c.set(JAVA_INT, CONFIG.byteOffset(MemoryLayout.PathElement.groupElement("psd_scaling")), psdScaling);
            c.set(JAVA_INT, CONFIG.byteOffset(MemoryLayout.PathElement.groupElement("psd_detrend")), psdDetrend);
            c.set(JAVA_INT, CONFIG.byteOffset(MemoryLayout.PathElement.groupElement("psd_precision")), psdPrecision);
            c.set(JAVA_INT, CONFIG.byteOffset(MemoryLayout.PathElement.groupElement("strict_reference")), strictReference ? 1 : 0);
            check((int) SET_CONFIG.invoke(engine, c));        // the engine copies the taps
        }
    }

    /**
     * The whole-recording waterfall straight from the data file (SigMfHelper.java:59-84: dataPath, headerBytes): no
     * mapped buffer, no 2 GiB limit (:78-82).  Rows of float32 dB, time-major.
     */
    public float[] spectrogramFromFile(String dataPath, long headerBytes, long firstSample, long frames, int fftSize,
                                       long hop, int window, String datatype) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int[] dt = parse(a, datatype);
            MemorySegment p = a.allocate(PARAMS);
            PARAMS_INIT.invoke(p);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("dtype")), dt[0]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("big_endian")), dt[1]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("window")), window);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("nfft")), fftSize);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("start_sample")), firstSample);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("hop")), hop);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("n_frames")), frames);
            MemorySegment out = a.allocate(ValueLayout.JAVA_FLOAT, frames * fftSize);
            check((int) SPECTROGRAM_FILE.invoke(engine, a.allocateFrom(dataPath), headerBytes, 0L, p, out, out.byteSize()));
            return out.toArray(ValueLayout.JAVA_FLOAT);
        }
    }

    /** Drop-in body of SpectralService.computeMagnitudes (SpectralService.java:33-85). */
    public double[] computeMagnitudes(MappedByteBuffer buffer, int startByte, int nfft, String datatype) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int[] dt = parse(a, datatype);
            MemorySegment out = a.allocate(JAVA_DOUBLE, nfft);
            MemorySegment seg = MemorySegment.ofBuffer(buffer);
            check((int) MAGNITUDES.invoke(engine, seg, seg.byteSize(), (long) startByte, nfft, dt[0], dt[1], out));
            return out.toArray(JAVA_DOUBLE);
        }
    }

    /** Replaces the whole `for t` loop of MainController.updateDisplay (MainController.java:980-999). */
    public double[][] computeWaterfall(MappedByteBuffer buffer, long currentSampleOffset, int canvasW, int fftSize,
                                       String datatype) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int[] dt = parse(a, datatype);
            MemorySegment p = a.allocate(PARAMS);
            PARAMS_INIT.invoke(p);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("dtype")), dt[0]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("big_endian")), dt[1]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("nfft")), fftSize);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("out_kind")), 1 /* SA_OUT_F64_DB */);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("start_sample")), currentSampleOffset);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("hop")), (long) fftSize);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("n_frames")), (long) canvasW);
            MemorySegment out = a.allocate(JAVA_DOUBLE, (long) canvasW * fftSize);
            MemorySegment seg = MemorySegment.ofBuffer(buffer);
            check((int) SPECTROGRAM.invoke(engine, seg, seg.byteSize(), p, out, out.byteSize()));
            double[][] waterfall = new double[canvasW][];
            for (int t = 0; t < canvasW; t++)
                waterfall[t] = out.asSlice((long) t * fftSize * 8, (long) fftSize * 8).toArray(JAVA_DOUBLE);
            return waterfall;
        }
    }

    /** Drop-in body of ExtractDownConvertService.extractAndDownConvert (ExtractDownConvertService.java:54-117). */
    public double[][] extractAndDownConvert(MappedByteBuffer buffer, long startSample, int count, String datatype,
                                            double freqOff, int down, boolean fast) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int[] dt = parse(a, datatype);
            long m = (long) DOWNCONVERT_LENGTH.invoke(engine, (long) count, down, fast ? 1 : 0);   // M under the engine's profile
            MemorySegment re = a.allocate(JAVA_DOUBLE, Math.max(m, 1)), im = a.allocate(JAVA_DOUBLE, Math.max(m, 1));
            MemorySegment len = a.allocate(JAVA_LONG);
            MemorySegment seg = MemorySegment.ofBuffer(buffer);
            check((int) DOWNCONVERT.invoke(engine, seg, seg.byteSize(), dt[0], dt[1], startSample, (long) count, freqOff,
                    down, fast ? 1 : 0, re, im, len));
            int n = (int) len.get(JAVA_LONG, 0);
            return new double[][] { re.asSlice(0, 8L * n).toArray(JAVA_DOUBLE), im.asSlice(0, 8L * n).toArray(JAVA_DOUBLE) };
        }
    }

    /**
     * ONE call for the batch loop of AnnotationController.executeCapability (AnnotationController.java:321-360, which
     * runs extractAndDownConvertAsync(...).join() per row): rows[i] = {startSample, count, freqOff, down}; fast = false
     * as at :336-337.  Returns the double[2][M_i] of every row and, when psdNfft > 0, the Welch PSD rows (dB, fs / down)
     * in psdOut[i] (psdOut may be null).  Only the annotated spans cross PCIe, once.
     */
    public double[][][] extractAndDownConvertBatch(MappedByteBuffer buffer, String datatype, double sampleRate,
                                                   double[][] rows, int psdNfft, double[][] psdOut) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int[] dt = parse(a, datatype);
            int n = rows.length;
            MemorySegment anns = a.allocate(ANNOTATION, n);
            MemorySegment offs = a.allocate(JAVA_LONG, Math.max(n, 1));
            long[] len = new long[n];
            long total = 0;
            for (int i = 0; i < n; i++) {
                long base = i * ANNOTATION.byteSize();
                anns.set(JAVA_LONG, base, (long) rows[i][0]);
                anns.set(JAVA_LONG, base + 8, (long) rows[i][1]);
                anns.set(JAVA_DOUBLE, base + 16, rows[i][2]);
                anns.set(JAVA_INT, base + 24, (int) rows[i][3]);
                anns.set(JAVA_INT, base + 28, 0);
                len[i] = (long) DOWNCONVERT_LENGTH.invoke(engine, (long) rows[i][1], (int) rows[i][3], 0);
                offs.setAtIndex(JAVA_LONG, i, total);
                total += 2 * len[i];
            }
            MemorySegment iq = a.allocate(JAVA_DOUBLE, Math.max(total, 1));
            MemorySegment psd = (psdNfft > 0 && psdOut != null) ? a.allocate(JAVA_DOUBLE, (long) n * psdNfft) : MemorySegment.NULL;
            MemorySegment seg = MemorySegment.ofBuffer(buffer);
            check((int) BATCH.invoke(engine, seg, seg.byteSize(), dt[0], dt[1], sampleRate, anns, n, psdNfft, 0L,
                    1 /* SA_WIN_HANN */, iq, offs, psd));
            double[][][] out = new double[n][][];
            for (int i = 0; i < n; i++) {
                long o = offs.getAtIndex(JAVA_LONG, i) * 8;
                out[i] = new double[][] { iq.asSlice(o, 8 * len[i]).toArray(JAVA_DOUBLE),
                                          iq.asSlice(o + 8 * len[i], 8 * len[i]).toArray(JAVA_DOUBLE) };
                if (psdNfft > 0 && psdOut != null) psdOut[i] = psd.asSlice((long) i * psdNfft * 8, (long) psdNfft * 8).toArray(JAVA_DOUBLE);
            }
            return out;
        }
    }

    /** Replaces PowerSpectralDensity.calculatePsdWelch at AnalysisDialogController.java:308-312 (any nfft <= data length). */
    public double[][] calculatePsdWelch(double[][] data, double fs, int nfft) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            MemorySegment re = a.allocateFrom(JAVA_DOUBLE, data[0]), im = a.allocateFrom(JAVA_DOUBLE, data[1]);
            MemorySegment f = a.allocate(JAVA_DOUBLE, nfft), db = a.allocate(JAVA_DOUBLE, nfft);
            check((int) PSD_WELCH.invoke(engine, re, im, (long) data[0].length, fs, nfft, 0L, 1 /* SA_WIN_HANN */, f, db));
            return new double[][] { f.toArray(JAVA_DOUBLE), db.toArray(JAVA_DOUBLE) };
        }
    }

    /**
     * MainController.renderSpectrogram (MainController.java:1261-1291) on the GPU: ARGB-ready RGBA8 bytes,
     * canvasH rows of canvasW pixels, row 0 = top.  The caller blits them with PixelWriter.setPixels.
     */
    public byte[] renderSpectrogram(MappedByteBuffer buffer, long currentSampleOffset, int canvasW, int canvasH,
                                    int fftSize, String datatype, double sampleRate, double minDb, double maxDb,
                                    int colormap) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int[] dt = parse(a, datatype);
            MemorySegment p = a.allocate(PARAMS);
            PARAMS_INIT.invoke(p);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("dtype")), dt[0]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("big_endian")), dt[1]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("nfft")), fftSize);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("start_sample")), currentSampleOffset);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("hop")), (long) fftSize);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("colormap")), colormap);
            p.set(JAVA_DOUBLE, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("sample_rate")), sampleRate);
            p.set(JAVA_DOUBLE, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("min_db")), minDb);
            p.set(JAVA_DOUBLE, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("max_db")), maxDb);
            MemorySegment out = a.allocate((long) canvasW * canvasH * 4);
            MemorySegment seg = MemorySegment.ofBuffer(buffer);
            check((int) RENDER_CANVAS.invoke(engine, seg, seg.byteSize(), p, canvasW, canvasH, 1L, 0 /* SA_REDUCE_NEAREST */, out));
            return out.toArray(ValueLayout.JAVA_BYTE);
        }
    }

    /**
     * Spectrum traces of a capture range (sa_spectrum_trace): the average (Welch PSD of the full band), peak-hold and
     * minimum-hold spectra of groups of framesPerRow frames, fft-shifted dB rows.  Returns {mean, max, min}, each
     * float[ceil(frames / framesPerRow)][fftSize], or null where the statistic was not wanted.
     */
    public float[][][] spectrumTrace(MappedByteBuffer buffer, long startSample, long frames, int fftSize, long hop,
                                     int window, String datatype, long framesPerRow, boolean mean, boolean max,
                                     boolean min) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int[] dt = parse(a, datatype);
            MemorySegment p = a.allocate(PARAMS);
            PARAMS_INIT.invoke(p);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("dtype")), dt[0]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("big_endian")), dt[1]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("window")), window);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("nfft")), fftSize);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("start_sample")), startSample);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("hop")), hop);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("n_frames")), frames);
            long rows = framesPerRow > 0 ? (frames + framesPerRow - 1) / framesPerRow : 0;
            long bytes = rows * fftSize * 4;
            boolean[] want = {mean, max, min};
            MemorySegment[] out = new MemorySegment[3];
            for (int s = 0; s < 3; s++) out[s] = want[s] ? a.allocate(Math.max(bytes, 4)) : MemorySegment.NULL;
            MemorySegment seg = MemorySegment.ofBuffer(buffer);
            check((int) SPECTRUM_TRACE.invoke(engine, seg, seg.byteSize(), p, framesPerRow, out[0], out[1], out[2], bytes));
            float[][][] res = new float[3][][];
            for (int s = 0; s < 3; s++) {
                if (!want[s]) continue;
                res[s] = new float[(int) rows][];
                for (int r = 0; r < rows; r++)
                    res[s][r] = out[s].asSlice((long) r * fftSize * 4, (long) fftSize * 4).toArray(ValueLayout.JAVA_FLOAT);
            }
            return res;
        }
    }

    /**
     * Persistence spectrum of a capture range (sa_spectrum_persistence): per fft-shifted bin, how many of the frames
     * landed on each of nLevels dB levels of [minDb, maxDb) (below the range: level 0, above it: the top level).
     * Returns int[nLevels][fftSize], level 0 the lowest; every column sums to frames.  The counts are UNSIGNED 32-bit
     * values held in Java ints: read them with Integer.toUnsignedLong when frames may exceed Integer.MAX_VALUE.
     */
    public int[][] spectrumPersistence(MappedByteBuffer buffer, long startSample, long frames, int fftSize, long hop,
                                       int window, String datatype, int nLevels, double minDb, double maxDb)
            throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int[] dt = parse(a, datatype);
            MemorySegment p = a.allocate(PARAMS);
            PARAMS_INIT.invoke(p);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("dtype")), dt[0]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("big_endian")), dt[1]);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("window")), window);
            p.set(JAVA_INT, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("nfft")), fftSize);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("start_sample")), startSample);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("hop")), hop);
            p.set(JAVA_LONG, PARAMS.byteOffset(MemoryLayout.PathElement.groupElement("n_frames")), frames);
            long bytes = (long) Math.max(nLevels, 0) * fftSize * 4;
            MemorySegment out = a.allocate(Math.max(bytes, 4));
            MemorySegment seg = MemorySegment.ofBuffer(buffer);
            check((int) SPECTRUM_PERSISTENCE.invoke(engine, seg, seg.byteSize(), p, nLevels, minDb, maxDb, out, bytes));
            int[][] res = new int[nLevels][];
            for (int l = 0; l < nLevels; l++)
                res[l] = out.asSlice((long) l * fftSize * 4, (long) fftSize * 4).toArray(ValueLayout.JAVA_INT);
            return res;
        }
    }

    /** Drop-in body of IqData.getInterleavedBinary (IqData.java:160-187). */
    public byte[] getInterleavedBinary(double[][] iqSamples, String format) throws Throwable {
        int code;
        if ("float32".equalsIgnoreCase(format)) code = 0;
        else if ("int16".equalsIgnoreCase(format)) code = 1;
        else throw new IllegalArgumentException("Unsupported binary format: " + format);
        try (Arena a = Arena.ofConfined()) {
            int n = iqSamples[0].length;
            MemorySegment re = a.allocateFrom(JAVA_DOUBLE, iqSamples[0]), im = a.allocateFrom(JAVA_DOUBLE, iqSamples[1]);
            MemorySegment out = a.allocate((long) n * (code == 0 ? 8 : 4));
            check((int) IQ_PACK.invoke(engine, re, im, (long) n, code, out));
            return out.toArray(ValueLayout.JAVA_BYTE);
        }
    }

    /**
     * The two O(N) loops of AnalysisDialogController.updateMagnitudeChart / updateFrequencyChart (:219-290):
     * returns {magnitude dB[n], smoothed instantaneous frequency + centre[n]} (element 0 of row 1 is NaN).
     */
    public double[][] analysisSeries(double[][] data, double sampleRate, double alphaMagn, double alphaFreq,
                                     double centerFreq) throws Throwable {
        try (Arena a = Arena.ofConfined()) {
            int n = data[0].length;
            MemorySegment re = a.allocateFrom(JAVA_DOUBLE, data[0]), im = a.allocateFrom(JAVA_DOUBLE, data[1]);
            MemorySegment mag = a.allocate(JAVA_DOUBLE, n), frq = a.allocate(JAVA_DOUBLE, n);
            check((int) ANALYSIS_SERIES.invoke(engine, re, im, (long) n, sampleRate, alphaMagn, alphaFreq, centerFreq, mag, frq));
            return new double[][] { mag.toArray(JAVA_DOUBLE), frq.toArray(JAVA_DOUBLE) };
        }
    }

    private static int[] parse(Arena a, String datatype) throws Throwable {
        MemorySegment d = a.allocate(JAVA_INT), be = a.allocate(JAVA_INT);
        check((int) PARSE_DT.invoke(a.allocateFrom(datatype), d, be));
        return new int[] { d.get(JAVA_INT, 0), be.get(JAVA_INT, 0) };
    }

    @Override public void close() {
        try { DESTROY.invoke(engine); } catch (Throwable ignored) { }
    }
}
