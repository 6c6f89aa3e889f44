// C++ consumer of the persistence spectrum: Engine::spectrumPersistence (include/sa_services.hpp) against the C entry
// sa_spectrum_persistence on the same request, plus its known answers (every column sums to the frame count; an
// on-bin tone puts every frame of its bin on one level).
#include <cmath>
#include <cstdio>
#include <cstring>
#include <vector>

#include "sa_services.hpp"

using namespace spectral_analyzer;

#define EXPECT(c) do { if (!(c)) { std::printf("FAIL %s:%d %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)

int main() {
    Engine eng(0);
    const int n = 1024, frames = 300, hop = 512, levels = 64;
    const size_t samples = (size_t)(frames - 2) * hop + n;           // the last frame is past the end of the buffer
    std::vector<float> iq(2 * samples);
    unsigned s = 12345;
    for (size_t i = 0; i < samples; i++) {
        const double ph = 2.0 * M_PI * 37.0 * (double)(i % n) / n;
        s = s * 1664525u + 1013904223u;
        const double noise = ((s >> 8) / 16777216.0 - 0.5) * 0.2;
        iq[2 * i] = (float)(std::cos(ph) + noise); iq[2 * i + 1] = (float)(std::sin(ph) - noise);
    }
    MappedByteBuffer buf{iq.data(), iq.size() * sizeof(float)};
    const std::vector<uint32_t> got = eng.spectrumPersistence(buf, "cf32_le", n, frames, hop, SA_WIN_HANN, 0, levels,
                                                              -120.0, 80.0);
    EXPECT(got.size() == (size_t)levels * n);
    const Datatype dt("cf32_le");
    sa_spectrogram_params p;
    sa_spectrogram_params_init(&p);
    p.dtype = dt.dtype; p.big_endian = dt.big_endian; p.nfft = n; p.hop = hop; p.window = SA_WIN_HANN; p.n_frames = frames;
    std::vector<uint32_t> ref((size_t)levels * n);
    EXPECT(sa_spectrum_persistence(eng.handle(), buf.data, buf.capacity, &p, levels, -120.0, 80.0, ref.data(),
                                   ref.size() * 4) == SA_OK);
    EXPECT(std::memcmp(got.data(), ref.data(), ref.size() * 4) == 0);
    for (int k = 0; k < n; k++) {
        uint64_t sum = 0;
        for (int l = 0; l < levels; l++) sum += got[(size_t)l * n + k];
        EXPECT(sum == (uint64_t)frames);
    }
    const int kt = (37 + n / 2) % n;                                  // fft-shifted tone bin
    int peak = 0;
    for (int l = 0; l < levels; l++) if (got[(size_t)l * n + kt] > got[(size_t)peak * n + kt]) peak = l;
    EXPECT(got[(size_t)peak * n + kt] == (uint32_t)(frames - 1));     // every readable frame on one level
    bool threw = false;
    try { eng.spectrumPersistence(buf, "cf32_le", n, frames, hop, SA_WIN_HANN, 0, 1, -120.0, 80.0); }
    catch (const std::exception&) { threw = true; }
    EXPECT(threw);                                                    // n_levels outside 2..256
    std::printf("cpp persistence ok\n");
    return 0;
}
