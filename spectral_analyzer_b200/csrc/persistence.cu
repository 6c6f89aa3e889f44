// persistence.cu -- persistence spectra of a capture range (sa_spectrum_persistence, include/sa_engine.h): per bin, how
// many frames of the spectrogram landed on each of n_levels dB levels.
//
// Frames and dB values d[t][k] are those of the spectrogram rows that sa_spectrogram_params describes (FP32 rows on FP32
// launches, FP64 rows on FP64 launches, eof_fill_db past the end of the buffer, -200 dB for strict-reference zero
// decodes).  In the launch's precision, each operation rounded on its own:
//   u = (d - min_db) * s,  s = n_levels / (max_db - min_db)   (min_db and s computed in FP64, rounded to the precision)
//   level = u >= 1 ? (int)min(u, n_levels - 1) : 0;   counts[level][(k + nfft/2) % nfft] += 1
// so the counts are exactly the histogram of the engine's own dB rows, and every column sums to n_frames.
//
// Two stages per chunk of frames:
//   1. the level instantiation (spectrogram_*_level_kernel, large_rows_level_kernel) of the transform kernel the
//      spectrogram dispatch picks (at 4096 points the mid kernel instead of radix-64, whose store code is its own)
//      writes OUT_LEVEL8 rows: one byte per bin, quantized from the db[] the F32 / F64 row stores would take, into a
//      chunk buffer;
//   2. persistence_hist_kernel counts the chunk's level rows into the histogram: each CTA owns a tile of up to 128 bins
//      x n_levels uint32 counters in shared memory, its warps walk a slab of frames, and the non-zero counters are
//      added into the global histogram with atomicAdd (integer addition: the result does not depend on their order).
// Chunk rule: a chunk holds min(n_frames, max(1, kLevelChunkBytes / nfft)) frames of level rows, kLevelChunkBytes =
// 512 MiB (the four-step workspace; 2^28 cf32 samples at 1024 points, hop 512, are one chunk).  DESIGN.md N5 has the
// measurement against chunks small enough to stay in L2.  The host entry streams the capture through the three-slot
// pipeline (H2D, stage 1 into the slot's output buffer, stage 2 into the one histogram); only the counts cross PCIe.
#include "engine_internal.h"

#include <algorithm>
#include <cmath>
#include <cstring>

using namespace sa;

namespace {

#ifndef SA_LEVEL_CHUNK_MB
#define SA_LEVEL_CHUNK_MB 512       // level rows per chunk of the device entry (a build-time constant for A/B runs)
#endif
constexpr uint64_t kLevelChunkBytes = (uint64_t)SA_LEVEL_CHUNK_MB << 20;
constexpr int kHistThreads = 1024;
constexpr int kHistUnroll = 8;                  // level rows in flight per warp
constexpr int kHistMaxLevels = 256;
constexpr uint64_t kHistMinSlab = 256;          // frames per CTA at least: the flush reads n_levels x tile counters

template <int BPL> struct LaneBytes;
template <> struct LaneBytes<2> { using V = unsigned short; };
template <> struct LaneBytes<4> { using V = unsigned int; };

// grid (nfft / TB tiles, slabs), TB = 32 * BPL bins.  Lane l of a warp takes bins [l BPL, (l + 1) BPL) of the tile in
// one load.  Counters are level-major, [level][slot] with slot j * 32 + l for the tile's bin l BPL + j, so the bank of
// every shared-memory atomic is its lane: the 32 lanes never collide, whatever levels they hold (a tone bin whose
// frames all land on one level included).
template <int BPL>
__global__ void __launch_bounds__(kHistThreads)
persistence_hist_kernel(const unsigned char* __restrict__ lv, const long long n_frames, const long long frames_per_slab,
                        const int nfft, const int n_levels, unsigned int* __restrict__ counts) {
    using V = typename LaneBytes<BPL>::V;
    constexpr int TB = 32 * BPL;
    extern __shared__ unsigned int hist[];
    for (int i = threadIdx.x; i < n_levels * TB; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const long long f0 = (long long)blockIdx.y * frames_per_slab;
    const long long f1 = min(n_frames, f0 + frames_per_slab);
    const unsigned char* base = lv + (size_t)blockIdx.x * TB + lane * BPL;
    unsigned int* hl = hist + lane;
    long long f = f0 + (threadIdx.x >> 5);
    for (; f + (long long)(kHistUnroll - 1) * nw < f1; f += (long long)kHistUnroll * nw) {
        unsigned int x[kHistUnroll];
#pragma unroll
        for (int u = 0; u < kHistUnroll; u++) x[u] = __ldcs(reinterpret_cast<const V*>(base + (size_t)(f + u * nw) * nfft));
#pragma unroll
        for (int u = 0; u < kHistUnroll; u++)
#pragma unroll
            for (int j = 0; j < BPL; j++) atomicAdd(&hl[((x[u] >> (8 * j)) & 255u) * TB + j * 32], 1u);
    }
    for (; f < f1; f += nw) {
        const unsigned int x = __ldcs(reinterpret_cast<const V*>(base + (size_t)f * nfft));
#pragma unroll
        for (int j = 0; j < BPL; j++) atomicAdd(&hl[((x >> (8 * j)) & 255u) * TB + j * 32], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n_levels * TB; i += blockDim.x) {
        const unsigned int c = hist[i];
        const int l = i / TB, s = i % TB;
        if (c) atomicAdd(&counts[(size_t)l * nfft + blockIdx.x * TB + (s % 32) * BPL + s / 32], c);
    }
}

// A validated request.
struct PersistPlan {
    sa_spectrogram_params p;          // out_kind = OUT_LEVEL8
    int prec = 0;
    LevelQuant q;
    uint64_t count_bytes = 0;         // n_levels * nfft uint32
};

int plan_persistence(const sa_spectrogram_params* params, uint32_t n_levels, double min_db, double max_db,
                     const void* out, uint64_t out_bytes, PersistPlan& t) {
    if (!params) return set_error(SA_ERR_INVALID_ARG, "params is NULL");
    // out_kind and the canvas fields (colormap, sample_rate, min_db, max_db) are ignored: validate the request as the
    // F32 rows it is counted from, so that canvas parameters reused here are not refused for their canvas fields
    sa_spectrogram_params p = *params;
    p.out_kind = SA_OUT_F32_DB;
    int rc = check_spec_params(&p, &t.prec);
    if (rc) return rc;
    if (n_levels < 2 || n_levels > kHistMaxLevels) return set_error(SA_ERR_INVALID_ARG, "n_levels %u outside 2..256", n_levels);
    if (!std::isfinite(min_db) || !std::isfinite(max_db) || !(max_db > min_db))
        return set_error(SA_ERR_INVALID_ARG, "the level range needs finite min_db < max_db");
    if (p.n_frames == 0) return set_error(SA_ERR_INVALID_ARG, "n_frames is 0");
    if (p.n_frames > 0xFFFFFFFFull) return set_error(SA_ERR_INVALID_ARG, "n_frames %llu does not fit the uint32 counts",
                                                     (unsigned long long)p.n_frames);
    if (!out) return set_error(SA_ERR_INVALID_ARG, "NULL output");
    t.p = p;
    t.p.out_kind = OUT_LEVEL8;
    t.q.min_db = min_db;
    t.q.scale = (double)n_levels / (max_db - min_db);
    t.q.n_levels = (int)n_levels;
    t.count_bytes = (uint64_t)n_levels * p.nfft * 4;
    if (out_bytes < t.count_bytes)
        return set_error(SA_ERR_SMALL_OUTPUT, "out_bytes %llu < %llu", (unsigned long long)out_bytes,
                         (unsigned long long)t.count_bytes);
    return SA_OK;
}

// the device quantizer (spectrogram_kernel.cuh db_level) on the host, for the constant levels of strict-zero requests
uint32_t host_level(double d, const PersistPlan& t) {
    const double top = (double)(t.q.n_levels - 1);
    if (t.prec == SA_PREC_F64) {
        const double u = (d - t.q.min_db) * t.q.scale;
        return u >= 1.0 ? (uint32_t)std::min(u, top) : 0;
    }
    const float df = (float)d, mn = (float)t.q.min_db, sc = (float)t.q.scale;
    const float diff = df - mn;
    const float u = diff * sc;
    return u >= 1.0f ? (uint32_t)std::min(u, (float)top) : 0;
}

// strict_zero requests: every readable frame holds -200 dB in every bin, every EOF frame eof_fill_db (readable frames
// are a prefix, MainController.java:987), so the histogram has at most two non-zero levels: n_read frames on level
// l_read and n_eof on level l_eof in every column.
struct StrictLevels { uint32_t l_read, n_read, l_eof, n_eof; };
StrictLevels strict_levels(const PersistPlan& t, uint64_t n_samples) {
    const sa_spectrogram_params& p = t.p;
    const uint64_t n_read = p.start_sample + p.nfft <= n_samples
                                ? std::min<uint64_t>(p.n_frames, (n_samples - p.start_sample - p.nfft) / p.hop + 1) : 0;
    return { host_level(-200.0, t), (uint32_t)n_read, host_level(p.eof_fill_db, t), (uint32_t)(p.n_frames - n_read) };
}

void strict_counts(const PersistPlan& t, uint64_t n_samples, uint32_t* counts) {
    const StrictLevels s = strict_levels(t, n_samples);
    const uint32_t nfft = t.p.nfft;
    std::fill_n(counts, (size_t)t.q.n_levels * nfft, 0u);
    for (uint32_t k = 0; k < nfft; k++) {
        counts[(size_t)s.l_read * nfft + k] += s.n_read;
        counts[(size_t)s.l_eof * nfft + k] += s.n_eof;
    }
}

// the same on the device, into zeroed counts (the device entry stays asynchronous); one thread per bin
__global__ void persistence_strict_kernel(uint32_t* counts, const int nfft, const StrictLevels s) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nfft) return;
    counts[(size_t)s.l_read * nfft + k] += s.n_read;
    counts[(size_t)s.l_eof * nfft + k] += s.n_eof;
}

// stage 2 over nf level rows at lv
int launch_hist(Engine* eng, const void* lv, uint64_t nf, const PersistPlan& t, uint32_t* d_counts, cudaStream_t stream) {
    const int nfft = (int)t.p.nfft, tb = std::min(128, nfft), nl = t.q.n_levels;
    const void* fn = tb == 128 ? (const void*)&persistence_hist_kernel<4> : (const void*)&persistence_hist_kernel<2>;
    const size_t smem = (size_t)nl * tb * 4;
    int& nb = eng->occupancy_smem[{fn, smem}];
    cudaError_t e = cudaSuccess;
    if (nb == 0) {                          // first launch of this (tile width, n_levels): attribute and occupancy
        e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, kHistMaxLevels * 128 * 4);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, kHistThreads, smem);
        if (e != cudaSuccess) { nb = 0; return cuda_fail(e, "persistence_hist_kernel occupancy"); }
        if (nb < 1) return set_error(SA_ERR_CUDA, "persistence_hist_kernel does not fit on an SM (smem %zu)", smem);
    }
    // CTAs of equal slabs: tiles x slabs fills whole waves of the resident slots, rounded down (a partial second wave of
    // full-length slabs would double the stage), unless the tiles alone take more than one wave
    const uint64_t tiles = (uint64_t)(nfft / tb), slots = (uint64_t)nb * eng->num_sms;
    const uint64_t waves = (tiles + slots - 1) / slots;
    const uint64_t want = waves * slots / tiles;
    const uint64_t cap = std::min<uint64_t>(65535, (nf + kHistMinSlab - 1) / kHistMinSlab);
    uint64_t slabs = std::max<uint64_t>(1, std::min(want, cap));
    long long fps = (long long)((nf + slabs - 1) / slabs);
    slabs = (nf + fps - 1) / fps;
    long long n = (long long)nf;
    int nfft_i = nfft, nl_i = nl;
    void* args[] = { (void*)&lv, &n, &fps, &nfft_i, &nl_i, &d_counts };
    e = cudaLaunchKernel(fn, dim3((unsigned)tiles, (unsigned)slabs), dim3(kHistThreads), args, smem, stream);
    if (e != cudaSuccess) return cuda_fail(e, "launch persistence_hist_kernel");
    eng->launches++;
    return SA_OK;
}

int persistence_device(Engine* eng, const void* d_iq, uint64_t n_samples, const PersistPlan& t, uint32_t* d_counts,
                       cudaStream_t stream) {
    const sa_spectrogram_params& p = t.p;
    cudaError_t e = cudaMemsetAsync(d_counts, 0, t.count_bytes, stream);
    if (e != cudaSuccess) return cuda_fail(e, "clear persistence counts");
    const uint64_t chunk = std::min<uint64_t>(p.n_frames, std::max<uint64_t>(1, kLevelChunkBytes / p.nfft));
    int rc = eng->ensure_scratch(12, chunk * p.nfft);
    if (rc) return rc;
    for (uint64_t f0 = 0; f0 < p.n_frames; f0 += chunk) {
        sa_spectrogram_params q = p;
        q.start_sample = p.start_sample + f0 * p.hop;
        q.n_frames = std::min<uint64_t>(chunk, p.n_frames - f0);
        rc = eng->launch_spectrogram(d_iq, n_samples, q, t.prec, eng->scratch[12], stream, 2, 0, 1, nullptr, &t.q);
        if (rc == SA_OK) rc = launch_hist(eng, eng->scratch[12], q.n_frames, t, d_counts, stream);
        if (rc) return rc;
    }
    eng->last_kernel += "+persistence_hist_kernel";
    return SA_OK;
}

// Host buffer: chunks of frames stream through the three pipeline slots (H2D -> level rows into the slot's output
// buffer -> histogram, on the slot's stream) into one device histogram; after the slots drain, one D2H of the counts.
int persistence_host(Engine* eng, const void* iq, uint64_t iq_bytes, const PersistPlan& t, uint32_t* out_counts) {
    const sa_spectrogram_params& p = t.p;
    const uint64_t bps = spec_bytes_per_iq(p);
    const uint64_t n_samples = iq_bytes / bps;
    // chunks bounded as the canvas path bounds them: the larger of the frames' level rows and their input samples
    const uint64_t per_frame = std::max<uint64_t>((uint64_t)p.nfft, p.hop * bps);
    const uint64_t fpc = std::min<uint64_t>(std::max<uint64_t>(1, eng->chunk_bytes / per_frame), p.n_frames);
    const uint64_t readable = n_samples > p.start_sample ? n_samples - p.start_sample : 0;
    const uint64_t in_cap = std::max<uint64_t>(16, std::min<uint64_t>((fpc - 1) * p.hop + p.nfft, readable) * bps);
    int rc = eng->ensure_scratch(12, t.count_bytes);
    if (rc) return rc;
    const bool in_pinned = host_ptr_is_pinned(iq);
    for (int i = 0; i < kSlots && rc == SA_OK; i++) {
        rc = eng->ensure_slot(eng->slots[i], in_cap, fpc * p.nfft);
        if (rc == SA_OK) rc = eng->ensure_staging(eng->slots[i], in_pinned ? 0 : in_cap, 0);
    }
    if (rc) return rc;
    auto drain = [&](int rc0) {             // nothing may be in flight on the staging buffers or the caller's memory
        for (int i = 0; i < kSlots; i++) {
            cudaError_t e = cudaStreamSynchronize(eng->slots[i].stream);
            if (e != cudaSuccess && rc0 == SA_OK) rc0 = cuda_fail(e, "persistence pipeline drain");
        }
        return rc0;
    };
    uint32_t* d_counts = static_cast<uint32_t*>(eng->scratch[12]);
    cudaStream_t s0 = eng->slots[0].stream;
    cudaError_t e = cudaMemsetAsync(d_counts, 0, t.count_bytes, s0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s0);              // before any slot's histogram adds to it
    if (e != cudaSuccess) return cuda_fail(e, "clear persistence counts");
    uint64_t c = 0;
    for (uint64_t f0 = 0; f0 < p.n_frames && rc == SA_OK; f0 += fpc, c++) {
        Slot& s = eng->slots[c % kSlots];
        e = cudaStreamSynchronize(s.stream);                          // slot buffers free again
        if (e != cudaSuccess) { rc = cuda_fail(e, "slot sync"); break; }
        const uint64_t nf = std::min<uint64_t>(fpc, p.n_frames - f0);
        const uint64_t s_begin = p.start_sample + f0 * p.hop;
        uint64_t s_end = s_begin + (nf - 1) * p.hop + p.nfft;
        if (s_end > n_samples) s_end = n_samples;                      // frames past EOF take eof_fill_db's level
        const uint64_t ns = s_end > s_begin ? s_end - s_begin : 0;
        if (ns) {
            const void* src = (const char*)iq + s_begin * bps;
            if (!in_pinned) { eng->host_copy(s.h_in, src, ns * bps); src = s.h_in; }
            e = cudaMemcpyAsync(s.d_in, src, ns * bps, cudaMemcpyHostToDevice, s.stream);
            if (e != cudaSuccess) { rc = cuda_fail(e, "H2D"); break; }
        }
        sa_spectrogram_params q = p;
        q.start_sample = 0;
        q.n_frames = nf;
        rc = eng->launch_spectrogram(s.d_in, ns, q, t.prec, s.d_out, s.stream, 5 + (int)(c % kSlots), 0, 1, nullptr, &t.q);
        if (rc == SA_OK) rc = launch_hist(eng, s.d_out, nf, t, d_counts, s.stream);
    }
    rc = drain(rc);
    if (rc) return rc;
    e = cudaMemcpyAsync(out_counts, d_counts, t.count_bytes, cudaMemcpyDeviceToHost, s0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s0);
    if (e != cudaSuccess) return cuda_fail(e, "D2H persistence counts");
    eng->last_kernel += "+persistence_hist_kernel";
    return SA_OK;
}

}  // namespace

extern "C" {

int32_t sa_spectrum_persistence(sa_engine* engine, const void* iq, uint64_t iq_bytes, const sa_spectrogram_params* params,
                                uint32_t n_levels, double min_db, double max_db, uint32_t* out_counts, uint64_t out_bytes) {
    ENGINE_ENTER(engine);
    PersistPlan t;
    int rc = plan_persistence(params, n_levels, min_db, max_db, out_counts, out_bytes, t);
    if (rc) return rc;
    if (!iq && iq_bytes) return set_error(SA_ERR_INVALID_ARG, "NULL buffer");
    if (strict_zero(t.p)) {                 // nothing is transformed: two levels from the frame counts
        strict_counts(t, iq_bytes / spec_bytes_per_iq(t.p), out_counts);
        engine->last_kernel = "none (strict_reference zero decode: constant persistence levels)";
        return SA_OK;
    }
    return persistence_host(engine, iq, iq_bytes, t, out_counts);
}

int32_t sa_spectrum_persistence_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes,
                                       const sa_spectrogram_params* params, uint32_t n_levels, double min_db,
                                       double max_db, uint32_t* d_counts, uint64_t out_bytes, void* cuda_stream) {
    ENGINE_ENTER(engine);
    PersistPlan t;
    int rc = plan_persistence(params, n_levels, min_db, max_db, d_counts, out_bytes, t);
    if (rc) return rc;
    if (!d_iq && iq_bytes) return set_error(SA_ERR_INVALID_ARG, "NULL buffer");
    const uint64_t bps = spec_bytes_per_iq(t.p);
    if ((uintptr_t)d_iq % bps) return set_error(SA_ERR_INVALID_ARG, "d_iq must be aligned to %llu bytes", (unsigned long long)bps);
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (strict_zero(t.p)) {                 // nothing is transformed: two levels from the frame counts, on the stream
        cudaError_t e = cudaMemsetAsync(d_counts, 0, t.count_bytes, stream);
        if (e != cudaSuccess) return cuda_fail(e, "clear persistence counts");
        const StrictLevels s = strict_levels(t, iq_bytes / bps);
        int nfft = (int)t.p.nfft;
        void* args[] = { &d_counts, &nfft, (void*)&s };
        e = cudaLaunchKernel((const void*)&persistence_strict_kernel, dim3((nfft + 255) / 256), dim3(256), args, 0, stream);
        if (e != cudaSuccess) return cuda_fail(e, "launch persistence_strict_kernel");
        engine->launches++;
        engine->last_kernel = "persistence_strict_kernel (strict_reference zero decode: constant persistence levels)";
        return SA_OK;
    }
    return persistence_device(engine, d_iq, iq_bytes / bps, t, d_counts, stream);
}

}  // extern "C"
