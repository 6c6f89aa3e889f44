// sa_services.hpp -- C++ host-side mirror of the reference's DSP service interface on top of the C-ABI
// (include/sa_engine.h).  Header-only.  The reference is compiled JVM code; its toolchain is absent from
// the build image, so this is the compiled-language host layer: same class and method names, argument
// meaning and error behaviour as the Java services it stands in for
//   SpectralService.computeMagnitudes                 S/services/SpectralService.java:33
//   ExtractDownConvertService.extractAndDownConvert   S/services/ExtractDownConvertService.java:34,54
//   PowerSpectralDensity.calculatePsdWelch [JDSP]     S/controllers/AnalysisDialogController.java:308-312
// (S/ = src/main/java/net/kcundercover/spectral_analyzer/).  Java exceptions map to C++ ones:
//   MathIllegalArgumentException -> std::invalid_argument, IndexOutOfBoundsException -> std::out_of_range.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <list>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "sa_engine.h"

namespace spectral_analyzer {

// The MappedByteBuffer of S/sigmf/SigMfHelper.java:78-84: a read-only view of the .sigmf-data bytes,
// position 0 already past core:header_bytes.
struct MappedByteBuffer {
    const void* data = nullptr;
    uint64_t capacity = 0;
};

inline void sa_check(int32_t rc) {
    if (rc == SA_OK) return;
    const std::string msg = sa_last_error();
    if (rc == SA_ERR_INVALID_ARG) throw std::invalid_argument(msg);
    if (rc == SA_ERR_OUT_OF_RANGE) throw std::out_of_range(msg);
    throw std::runtime_error("sa_engine error " + std::to_string(rc) + ": " + msg);
}

class Engine {
public:
    explicit Engine(int device = 0) { sa_check(sa_engine_create(device, &h_)); }
    ~Engine() { sa_engine_destroy(h_); }
    Engine(const Engine&) = delete;
    Engine& operator=(const Engine&) = delete;
    sa_engine* handle() const { return h_; }
    // anonymous memory only: cudaHostRegister refuses file-backed mappings (the engine stages those itself)
    void registerHost(const MappedByteBuffer& b) { sa_check(sa_register_host(h_, b.data, b.capacity, 1)); }
    void unregisterHost(const MappedByteBuffer& b) { sa_check(sa_unregister_host(h_, b.data)); }
    // the engine's JDSP profile (sa_analysis_config: taps, delay / length rule, PSD scaling / detrend / precision)
    void setAnalysisConfig(const sa_analysis_config& c) { sa_check(sa_set_analysis_config(h_, &c)); }
    void resetAnalysisConfig() { sa_check(sa_set_analysis_config(h_, nullptr)); }
    // spectrum traces (sa_spectrum_trace): average / peak-hold / minimum-hold spectra of groups of framesPerRow frames
    // of the spectrogram these arguments describe; each wanted statistic is float [ceil(frames / framesPerRow)][fftSize]
    // fft-shifted dB, the others stay empty
    struct Traces { std::vector<float> mean, max, min; };
    Traces spectrumTrace(const MappedByteBuffer& buffer, const std::string& datatype, int fftSize, int64_t frames,
                         int64_t hop, int window, int64_t startSample, int64_t framesPerRow, bool wantMean = true,
                         bool wantMax = true, bool wantMin = false) const;
    // persistence spectrum (sa_spectrum_persistence): per fft-shifted bin, how many of the frames of the spectrogram
    // these arguments describe landed on each of nLevels dB levels of [minDb, maxDb); uint32 [nLevels][fftSize],
    // level 0 the lowest, every column summing to frames
    std::vector<uint32_t> spectrumPersistence(const MappedByteBuffer& buffer, const std::string& datatype, int fftSize,
                                              int64_t frames, int64_t hop, int window, int64_t startSample, int nLevels,
                                              double minDb, double maxDb) const;
private:
    sa_engine* h_ = nullptr;
};

struct Datatype {
    int32_t dtype = 0, big_endian = 0;
    explicit Datatype(const std::string& sigmf) { sa_check(sa_parse_datatype(sigmf.c_str(), &dtype, &big_endian)); }
};

inline Engine::Traces Engine::spectrumTrace(const MappedByteBuffer& buffer, const std::string& datatype, int fftSize,
                                            int64_t frames, int64_t hop, int window, int64_t startSample,
                                            int64_t framesPerRow, bool wantMean, bool wantMax, bool wantMin) const {
    const Datatype dt(datatype);
    sa_spectrogram_params p;
    sa_spectrogram_params_init(&p);
    p.dtype = dt.dtype; p.big_endian = dt.big_endian; p.nfft = (uint32_t)fftSize; p.hop = (uint64_t)hop;
    p.window = window; p.start_sample = (uint64_t)startSample; p.n_frames = (uint64_t)frames;
    const size_t n = framesPerRow > 0 ? (size_t)((frames + framesPerRow - 1) / framesPerRow) * (size_t)fftSize : 0;
    Traces t;
    if (wantMean) t.mean.resize(n);
    if (wantMax) t.max.resize(n);
    if (wantMin) t.min.resize(n);
    sa_check(sa_spectrum_trace(h_, buffer.data, buffer.capacity, &p, (uint64_t)framesPerRow, wantMean ? t.mean.data() : nullptr,
                               wantMax ? t.max.data() : nullptr, wantMin ? t.min.data() : nullptr, n * sizeof(float)));
    return t;
}

inline std::vector<uint32_t> Engine::spectrumPersistence(const MappedByteBuffer& buffer, const std::string& datatype,
                                                         int fftSize, int64_t frames, int64_t hop, int window,
                                                         int64_t startSample, int nLevels, double minDb,
                                                         double maxDb) const {
    const Datatype dt(datatype);
    sa_spectrogram_params p;
    sa_spectrogram_params_init(&p);
    p.dtype = dt.dtype; p.big_endian = dt.big_endian; p.nfft = (uint32_t)fftSize; p.hop = (uint64_t)hop;
    p.window = window; p.start_sample = (uint64_t)startSample; p.n_frames = (uint64_t)frames;
    std::vector<uint32_t> counts(nLevels > 0 && fftSize > 0 ? (size_t)nLevels * (size_t)fftSize : 0);
    sa_check(sa_spectrum_persistence(h_, buffer.data, buffer.capacity, &p, (uint32_t)nLevels, minDb, maxDb, counts.data(),
                                     counts.size() * sizeof(uint32_t)));
    return counts;
}

class SpectralService {
public:
    explicit SpectralService(Engine& e) : e_(e) {}
    // double[] computeMagnitudes(MappedByteBuffer buffer, int startByte, int nfft, String datatype)
    std::vector<double> computeMagnitudes(const MappedByteBuffer& buffer, int startByte, int nfft,
                                          const std::string& datatype) const {
        const Datatype dt(datatype);
        std::vector<double> out((size_t)nfft);
        sa_check(sa_compute_magnitudes(e_.handle(), buffer.data, buffer.capacity, (uint64_t)startByte, (uint32_t)nfft,
                                       dt.dtype, dt.big_endian, out.data()));
        return out;
    }
    // The same waterfall read from the data file itself (SigMfHelper.load, S/sigmf/SigMfHelper.java:59-84: dataPath and
    // core:header_bytes): parallel pread into the engine's pinned ring, no mapped buffer and no 2 GiB limit.
    std::vector<float> computeWaterfallFromFile(const std::string& dataPath, uint64_t headerBytes, int64_t firstSample,
                                                int64_t frames, int fftSize, int64_t hop, int window,
                                                const std::string& datatype) const {
        const Datatype dt(datatype);
        sa_spectrogram_params p;
        sa_spectrogram_params_init(&p);
        p.dtype = dt.dtype; p.big_endian = dt.big_endian; p.nfft = (uint32_t)fftSize; p.hop = (uint64_t)hop;
        p.window = window; p.start_sample = (uint64_t)firstSample; p.n_frames = (uint64_t)frames;
        std::vector<float> out((size_t)frames * fftSize);
        sa_check(sa_spectrogram_file(e_.handle(), dataPath.c_str(), headerBytes, 0, &p, out.data(), out.size() * sizeof(float)));
        return out;
    }
    // The frame loop of MainController.updateDisplay (:980-999) as one call: waterfall[canvasW][fftSize].
    std::vector<double> computeWaterfall(const MappedByteBuffer& buffer, int64_t currentSampleOffset, int canvasW,
                                         int fftSize, const std::string& datatype) const {
        const Datatype dt(datatype);
        sa_spectrogram_params p;
        sa_spectrogram_params_init(&p);
        p.dtype = dt.dtype; p.big_endian = dt.big_endian; p.nfft = (uint32_t)fftSize; p.hop = (uint64_t)fftSize;
        p.start_sample = (uint64_t)currentSampleOffset; p.n_frames = (uint64_t)canvasW; p.out_kind = SA_OUT_F64_DB;
        std::vector<double> out((size_t)canvasW * fftSize);
        sa_check(sa_spectrogram(e_.handle(), buffer.data, buffer.capacity, &p, out.data(), out.size() * sizeof(double)));
        return out;
    }
private:
    Engine& e_;
};

class ExtractDownConvertService {
public:
    explicit ExtractDownConvertService(Engine& e) : e_(e) {}
    // double[2][M] extractAndDownConvert(buffer, long startSample, int count, String datatype,
    //                                    double freqOff, int down, boolean fast = false)
    std::vector<std::vector<double>> extractAndDownConvert(const MappedByteBuffer& buffer, int64_t startSample, int count,
                                                           const std::string& datatype, double freqOff, int down,
                                                           bool fast = false) const {
        const Datatype dt(datatype);
        if (down < 1) throw std::invalid_argument("down < 1");
        const size_t m = (size_t)sa_downconvert_length(e_.handle(), (uint64_t)count, down, fast ? 1 : 0);
        std::vector<std::vector<double>> out(2, std::vector<double>(m ? m : 1));
        uint64_t n = 0;
        sa_check(sa_downconvert(e_.handle(), buffer.data, buffer.capacity, dt.dtype, dt.big_endian, (uint64_t)startSample,
                                (uint64_t)count, freqOff, down, fast ? 1 : 0, out[0].data(), out[1].data(), &n));
        out[0].resize(n); out[1].resize(n);
        return out;
    }
    // The batch loop of AnnotationController.executeCapability (S/controllers/AnnotationController.java:321-360: one
    // extractAndDownConvertAsync(..., fast = false).join() per selected row) as ONE call: only the annotated spans cross
    // PCIe, once.  Returns the double[2][M_i] of every annotation; when psdNfft > 0 the Welch PSD rows (dB, sampling
    // rate sampleRate / down, fft-shifted; shorter annotations follow the caller's single-window rule, rest of the row
    // NaN) are written to *psd as [n][psdNfft].
    struct Annotation { int64_t startSample; int count; double freqOff; int down; };
    std::vector<std::vector<std::vector<double>>> extractAndDownConvertBatch(
            const MappedByteBuffer& buffer, const std::string& datatype, double sampleRate,
            const std::vector<Annotation>& rows, int psdNfft = 0, std::vector<double>* psd = nullptr) const {
        const Datatype dt(datatype);
        std::vector<sa_annotation> anns(rows.size());
        std::vector<uint64_t> offs(rows.size()), len(rows.size());
        uint64_t total = 0;
        for (size_t i = 0; i < rows.size(); i++) {
            if (rows[i].down < 1) throw std::invalid_argument("down < 1");
            anns[i].start_sample = (uint64_t)rows[i].startSample; anns[i].count = (uint64_t)rows[i].count;
            anns[i].freq_off = rows[i].freqOff; anns[i].down = rows[i].down; anns[i].fast = 0;
            len[i] = sa_downconvert_length(e_.handle(), anns[i].count, anns[i].down, 0);
            offs[i] = total;
            total += 2 * len[i];
        }
        std::vector<double> iq(total ? total : 1);
        const bool want_psd = psdNfft > 0 && psd != nullptr;
        if (want_psd) psd->assign(rows.size() * (size_t)psdNfft, 0.0);
        sa_check(sa_downconvert_psd_batch(e_.handle(), buffer.data, buffer.capacity, dt.dtype, dt.big_endian, sampleRate,
                                          anns.data(), (uint32_t)anns.size(), want_psd ? (uint32_t)psdNfft : 0, 0,
                                          SA_WIN_HANN, iq.data(), offs.data(), want_psd ? psd->data() : nullptr));
        std::vector<std::vector<std::vector<double>>> out(rows.size());
        for (size_t i = 0; i < rows.size(); i++) {
            const double* p = iq.data() + offs[i];
            out[i] = { std::vector<double>(p, p + len[i]), std::vector<double>(p + len[i], p + 2 * len[i]) };
        }
        return out;
    }
private:
    Engine& e_;
};

struct PowerSpectralDensity {
    // double[2][K] calculatePsdWelch(double[][] data, double fs, int nfft): row 0 = frequency axis centred on 0,
    // row 1 = level in dB/Hz
    static std::vector<std::vector<double>> calculatePsdWelch(Engine& e, const std::vector<std::vector<double>>& data,
                                                              double fs, int nfft) {
        std::vector<std::vector<double>> out(2, std::vector<double>((size_t)nfft));
        sa_check(sa_psd_welch(e.handle(), data[0].data(), data[1].data(), data[0].size(), fs, (uint32_t)nfft, 0,
                              SA_WIN_HANN, out[0].data(), out[1].data()));
        return out;
    }
};

// MainController.renderSpectrogram (S/controllers/MainController.java:1261-1291) for a canvasW x canvasH view:
// RGBA8 [canvasH][canvasW], row 0 = top.  framesPerColumn = 1 / SA_REDUCE_NEAREST is the reference.
struct SpectrogramRenderer {
    static std::vector<uint8_t> renderSpectrogram(Engine& e, const MappedByteBuffer& buffer, int64_t currentSampleOffset,
                                                  int canvasW, int canvasH, int fftSize, const std::string& datatype,
                                                  double sampleRate, double minDb, double maxDb, int colormap,
                                                  int64_t framesPerColumn = 1, int reduce = SA_REDUCE_NEAREST) {
        const Datatype dt(datatype);
        sa_spectrogram_params p;
        sa_spectrogram_params_init(&p);
        p.dtype = dt.dtype; p.big_endian = dt.big_endian; p.nfft = (uint32_t)fftSize; p.hop = (uint64_t)fftSize;
        p.start_sample = (uint64_t)currentSampleOffset; p.sample_rate = sampleRate; p.min_db = minDb; p.max_db = maxDb;
        p.colormap = colormap;
        std::vector<uint8_t> out((size_t)canvasW * canvasH * 4);
        sa_check(sa_render_canvas(e.handle(), buffer.data, buffer.capacity, &p, (uint32_t)canvasW, (uint32_t)canvasH,
                                  (uint64_t)framesPerColumn, reduce, out.data()));
        return out;
    }
};

// Scrolling views: the reference redraws every column on each scroll-bar move (MainController.java:319 -> :980-999).
// A view is assembled from fixed-width tiles of canvas columns kept in an LRU map, so that a scroll step renders
// only the tiles that enter the view (same scheme as spectral_analyzer_b200/tiles.py).  Tiles are aligned on global
// column indices of the view's phase (start % samples-per-column); the result is bit-identical to one
// renderSpectrogram call at the same start.
class CanvasTileCache {
public:
    CanvasTileCache(Engine& e, int tileW = 256, size_t maxTiles = 64) : e_(e), tileW_(tileW), maxTiles_(maxTiles) {
        if (tileW < 1 || maxTiles < 1) throw std::invalid_argument("tileW and maxTiles must be positive");
    }
    size_t hits() const { return hits_; }
    size_t misses() const { return misses_; }
    void clear() { lru_.clear(); index_.clear(); }

    std::vector<uint8_t> view(const MappedByteBuffer& buffer, int64_t currentSampleOffset, int canvasW, int canvasH,
                              int fftSize, const std::string& datatype, double sampleRate, double minDb, double maxDb,
                              int colormap, int64_t framesPerColumn = 1, int reduce = SA_REDUCE_NEAREST) {
        if (currentSampleOffset < 0) throw std::invalid_argument("currentSampleOffset must be non-negative");
        const int64_t spc = framesPerColumn * (int64_t)fftSize;
        const int64_t phase = currentSampleOffset % spc, g0 = currentSampleOffset / spc;
        std::vector<uint8_t> out((size_t)canvasW * canvasH * 4);
        for (int64_t k = g0 / tileW_; k <= (g0 + canvasW - 1) / tileW_; k++) {
            char key[256];
            std::snprintf(key, sizeof(key), "%p/%llu/%s/%d/%d/%lld/%d/%d/%.17g/%.17g/%.17g/%lld/%lld", buffer.data,
                          (unsigned long long)buffer.capacity, datatype.c_str(), fftSize, canvasH, (long long)framesPerColumn,
                          reduce, colormap, minDb, maxDb, sampleRate, (long long)phase, (long long)k);
            auto it = index_.find(key);
            if (it == index_.end()) {
                misses_++;
                lru_.emplace_front(key, SpectrogramRenderer::renderSpectrogram(
                    e_, buffer, phase + k * tileW_ * spc, tileW_, canvasH, fftSize, datatype, sampleRate, minDb, maxDb,
                    colormap, framesPerColumn, reduce));
                index_[key] = lru_.begin();
                while (lru_.size() > maxTiles_) { index_.erase(lru_.back().first); lru_.pop_back(); }
                it = index_.find(key);
            } else {
                hits_++;
                lru_.splice(lru_.begin(), lru_, it->second);
            }
            const std::vector<uint8_t>& tile = it->second->second;
            const int64_t lo = std::max<int64_t>(g0, k * tileW_), hi = std::min<int64_t>(g0 + canvasW, (k + 1) * tileW_);
            for (int y = 0; y < canvasH; y++)
                std::memcpy(&out[((size_t)y * canvasW + (size_t)(lo - g0)) * 4],
                            &tile[((size_t)y * tileW_ + (size_t)(lo - k * tileW_)) * 4], (size_t)(hi - lo) * 4);
        }
        return out;
    }
private:
    using Entry = std::pair<std::string, std::vector<uint8_t>>;
    Engine& e_;
    int tileW_;
    size_t maxTiles_, hits_ = 0, misses_ = 0;
    std::list<Entry> lru_;
    std::unordered_map<std::string, std::list<Entry>::iterator> index_;
};

// S/data/IqData.java: the binary packers of the downconverted double[2][N] (getInterleavedBinary :160-187)
class IqData {
public:
    IqData(Engine& e, std::vector<std::vector<double>> iqSamples) : e_(e), iq_(std::move(iqSamples)) {}
    std::vector<uint8_t> getInterleavedBinary(const std::string& format) const {
        int code;
        if (format == "float32" || format == "FLOAT32") code = SA_PACK_F32;
        else if (format == "int16" || format == "INT16") code = SA_PACK_I16;
        else throw std::invalid_argument("Unsupported binary format: " + format);
        std::vector<uint8_t> out(iq_[0].size() * (code == SA_PACK_F32 ? 8 : 4));
        sa_check(sa_iq_pack(e_.handle(), iq_[0].data(), iq_[1].data(), iq_[0].size(), code, out.data()));
        return out;
    }
private:
    Engine& e_;
    std::vector<std::vector<double>> iq_;
};

}  // namespace spectral_analyzer
