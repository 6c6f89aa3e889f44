// trace.cu -- spectrum traces of a capture range (sa_spectrum_trace, include/sa_engine.h): the average (Welch PSD of
// the full band), peak-hold and minimum-hold spectra of groups of frames_per_row frames, reduced in the spectrogram
// epilogue.
//
// Frames are those of the spectrogram that sa_spectrogram_params describes.  Output row r reduces frames
// [r F, min((r + 1) F, n_frames)), F = frames_per_row; per frame t and bin k, P_t[k] = |X_t[k]|^2 (0 for a strict-reference
// decode that yields zeros), or for a frame past the end of the buffer the power whose level is eof_fill_db.
//   MEAN = sum P / count (EOF frames counted), MAX = max P, MIN = min P,
// each written as the level 20 log10(sqrt(P) + 1e-10) (SA_DB_MAG_1E10) or 10 log10(P + 1e-20) (SA_DB_POWER).
//
// Two stages:
//   1. the transform kernel the spectrogram dispatch picks (pool_mode POOL_TRACE; at 4096 points the mid kernel instead
//      of radix-64, whose store code is its own) reduces |X|^2 of every frame into accumulator cells: one red per wanted
//      statistic, bin and frame, 32 consecutive bins per warp instruction.  A cell holds at most kTraceCellFrames = 256
//      frames of one row, in the launch's precision (FP32 / FP64).  So an FP32 cell sums at most 256 non-negative terms,
//      the atomics spread over cells x nfft addresses instead of nfft, and only the order inside a cell can vary.
//   2. trace_finalize_kernel combines each row's cells in FP64 in a fixed order (sum / count, max, min), takes the level
//      in FP64 and writes F32 / F64 rows: MAX and MIN are bit-reproducible, MEAN varies only inside a cell.
// The host entry streams the capture through the three-slot pipeline; every chunk reduces into the same accumulator
// (atomics, so chunks need no alignment to cells), and only the trace rows cross PCIe.  Requests whose accumulator
// would exceed kTraceAccBytes run in groups of whole rows.
#include "engine_internal.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

using namespace sa;

namespace {

constexpr uint64_t kTraceAccBytes = 1ull << 30;   // accumulator cells of one group of rows
constexpr int kFinalizeBins = 32;                 // bins per finalize block (one 128-byte line of FP32 cells)
constexpr int kFinalizeGroups = 32;               // cell groups per finalize block at most

struct TraceFinalizeArgs {
    const void* acc[3];     // sum, max, min cells [row][cpr][nfft] of this group (nullptr = not wanted)
    void* out[3];           // rows of this group [row][nfft], F32 or F64
    long long cpr;          // cells per row
    long long fpr;          // frames per row
    long long n_frames;     // frames of this group: row r counts min(fpr, n_frames - r fpr)
    int nfft;
    int out_f64;
    int db_mode;
};

__device__ __forceinline__ double trace_level(double p, int db_mode) {
    return db_mode == DBM_MAG_1E10 ? 20.0 * log10(sqrt(p) + 1e-10) : 10.0 * log10(p + 1e-20);
}

template <typename A> struct AccBits;
template <> struct AccBits<float> {
    using U = unsigned int;
    static __device__ __forceinline__ double val(U b) { return (double)__uint_as_float(b); }
};
template <> struct AccBits<double> {
    using U = unsigned long long;
    static __device__ __forceinline__ double val(U b) { return __longlong_as_double((long long)b); }
};

// block (kFinalizeBins bins, G cell groups), grid (nfft / kFinalizeBins, rows).  Group g combines the cells
// [g cpr / G, (g + 1) cpr / G) of its row in ascending order, then thread row 0 combines the G partials in ascending
// order: a fixed order, whatever the launch.
template <typename A>
__global__ void __launch_bounds__(kFinalizeBins * kFinalizeGroups)
trace_finalize_kernel(const TraceFinalizeArgs a) {
    using U = typename AccBits<A>::U;
    __shared__ double s_sum[kFinalizeGroups][kFinalizeBins];
    __shared__ U s_max[kFinalizeGroups][kFinalizeBins], s_min[kFinalizeGroups][kFinalizeBins];
    const int k = blockIdx.x * kFinalizeBins + threadIdx.x;
    const long long row = blockIdx.y;
    const int g = threadIdx.y, G = blockDim.y;
    const long long c0 = row * a.cpr + (long long)g * a.cpr / G, c1 = row * a.cpr + (long long)(g + 1) * a.cpr / G;
    const A* sum_p = reinterpret_cast<const A*>(a.acc[0]);
    const U* max_p = reinterpret_cast<const U*>(a.acc[1]);
    const U* min_p = reinterpret_cast<const U*>(a.acc[2]);
    double sum = 0.0;
    U mx = 0, mnc = 0;                          // MIN cells hold the complement of the bit pattern
#pragma unroll 4
    for (long long c = c0; c < c1; c++) {
        const size_t i = (size_t)c * a.nfft + k;
        if (sum_p) sum += (double)__ldcg(&sum_p[i]);
        if (max_p) mx = max(mx, __ldcg(&max_p[i]));
        if (min_p) mnc = max(mnc, __ldcg(&min_p[i]));
    }
    s_sum[g][threadIdx.x] = sum; s_max[g][threadIdx.x] = mx; s_min[g][threadIdx.x] = mnc;
    __syncthreads();
    if (g != 0) return;
    for (int j = 1; j < G; j++) {
        sum += s_sum[j][threadIdx.x];
        mx = max(mx, s_max[j][threadIdx.x]);
        mnc = max(mnc, s_min[j][threadIdx.x]);
    }
    const long long cnt = min(a.fpr, a.n_frames - row * a.fpr);
    const double v[3] = { sum / (double)cnt, AccBits<A>::val(mx), AccBits<A>::val((U)~mnc) };
    const size_t o = (size_t)row * a.nfft + k;
#pragma unroll
    for (int s = 0; s < 3; s++) {
        if (!a.out[s]) continue;
        const double lv = trace_level(v[s], a.db_mode);
        if (a.out_f64) reinterpret_cast<double*>(a.out[s])[o] = lv;
        else reinterpret_cast<float*>(a.out[s])[o] = (float)lv;
    }
}

// A validated request and its accumulator geometry.
struct TracePlan {
    sa_spectrogram_params p;
    int prec = 0;
    uint64_t fpr = 0;                 // frames per row, at most n_frames
    uint64_t n_rows = 0;
    uint64_t cpr = 0, kc = 0;         // cells per row, frames per cell
    uint64_t acc_elem = 0;            // 4 (FP32 launches) or 8 (FP64)
    uint64_t out_elem = 0;
    int nstats = 0;
    int stat_of[3] = {-1, -1, -1};    // statistic -> accumulator slot
    uint64_t rows_per_group = 0;
    uint64_t cell_bytes() const { return cpr * p.nfft * acc_elem; }                 // one row, one statistic
};

int plan_trace(const sa_spectrogram_params* params, uint64_t frames_per_row, void* const outs[3], uint64_t out_bytes,
               TracePlan& t) {
    int rc = check_spec_params(params, &t.prec);
    if (rc) return rc;
    const sa_spectrogram_params& p = *params;
    if (frames_per_row == 0) return set_error(SA_ERR_INVALID_ARG, "frames_per_row is 0");
    if (p.n_frames == 0) return set_error(SA_ERR_INVALID_ARG, "n_frames is 0");
    if (!outs[0] && !outs[1] && !outs[2]) return set_error(SA_ERR_INVALID_ARG, "no statistic wanted (all outputs NULL)");
    if (p.out_kind == SA_OUT_RGBA8) return set_error(SA_ERR_INVALID_ARG, "a trace is written as F32 or F64 dB, not RGBA8");
    t.p = p;
    t.fpr = std::min<uint64_t>(frames_per_row, p.n_frames);          // rows of more frames than exist: one row
    t.n_rows = p.n_frames / t.fpr + (p.n_frames % t.fpr != 0);
    t.out_elem = p.out_kind == SA_OUT_F64_DB ? 8 : 4;
    const uint64_t need = t.n_rows * p.nfft * t.out_elem;
    if (out_bytes < need)
        return set_error(SA_ERR_SMALL_OUTPUT, "out_bytes %llu < %llu", (unsigned long long)out_bytes, (unsigned long long)need);
    t.kc = std::min<uint64_t>(t.fpr, kTraceCellFrames);
    t.cpr = (t.fpr + t.kc - 1) / t.kc;
    t.acc_elem = t.prec == SA_PREC_F64 ? 8 : 4;
    for (int s = 0; s < 3; s++) if (outs[s]) t.stat_of[s] = t.nstats++;
    const uint64_t row_bytes = t.cell_bytes() * t.nstats;
    if (row_bytes > kTraceAccBytes)
        return set_error(SA_ERR_UNSUPPORTED, "one trace row needs %llu bytes of accumulator cells (more than %llu)",
                         (unsigned long long)row_bytes, (unsigned long long)kTraceAccBytes);
    t.rows_per_group = std::min<uint64_t>(std::min<uint64_t>(t.n_rows, 65535), kTraceAccBytes / row_bytes);
    return SA_OK;
}

double host_level(double p, int db_mode) {
    return db_mode == SA_DB_MAG_1E10 ? 20.0 * std::log10(std::sqrt(p) + 1e-10) : 10.0 * std::log10(p + 1e-20);
}

// strict_zero requests: every readable frame has P = 0, every EOF frame the EOF power, so each row is a constant
// given by its counts of readable and EOF frames (readable frames are a prefix, MainController.java:987).
// rows: n_rows * nfft elements of out_kind per wanted statistic.
void strict_trace_rows(const TracePlan& t, uint64_t n_samples, void* const outs[3]) {
    const sa_spectrogram_params& p = t.p;
    const uint64_t n_read = p.start_sample + p.nfft <= n_samples
                                ? std::min<uint64_t>(p.n_frames, (n_samples - p.start_sample - p.nfft) / p.hop + 1) : 0;
    const double pe = eof_power(p);
    for (uint64_t r = 0; r < t.n_rows; r++) {
        const uint64_t f0 = r * t.fpr, cnt = std::min<uint64_t>(t.fpr, p.n_frames - f0);
        const uint64_t nr = n_read > f0 ? std::min<uint64_t>(cnt, n_read - f0) : 0, ne = cnt - nr;
        const double v[3] = { (double)ne * pe / (double)cnt, ne ? pe : 0.0, nr ? 0.0 : pe };
        for (int s = 0; s < 3; s++) {
            if (!outs[s]) continue;
            const double lv = host_level(v[s], p.db_mode);
            if (t.out_elem == 8) std::fill_n((double*)outs[s] + r * p.nfft, p.nfft, lv);
            else std::fill_n((float*)outs[s] + r * p.nfft, p.nfft, (float)lv);
        }
    }
}

// accumulator cells of the group starting at row g0 (nr rows), in scratch[10]
void group_cells(Engine* eng, const TracePlan& t, TraceCells& tc) {
    const uint64_t stride = t.rows_per_group * t.cell_bytes();
    for (int s = 0; s < 3; s++)
        tc.acc[s] = t.stat_of[s] < 0 ? nullptr : (char*)eng->scratch[10] + t.stat_of[s] * stride;
    tc.frame0 = 0;
    tc.cells_per_row = t.cpr;
    tc.frames_per_cell = t.kc;
}

int launch_finalize(Engine* eng, const TracePlan& t, const TraceCells& tc, uint64_t group_frames, uint64_t nr,
                    void* const outs[3], uint64_t out_row0, cudaStream_t stream) {
    TraceFinalizeArgs fa;
    memset(&fa, 0, sizeof(fa));
    for (int s = 0; s < 3; s++) {
        fa.acc[s] = tc.acc[s];
        fa.out[s] = outs[s] ? (char*)outs[s] + out_row0 * t.p.nfft * t.out_elem : nullptr;
    }
    fa.cpr = (long long)t.cpr;
    fa.fpr = (long long)t.fpr;
    fa.n_frames = (long long)group_frames;
    fa.nfft = (int)t.p.nfft;
    fa.out_f64 = t.out_elem == 8;
    fa.db_mode = t.p.db_mode;
    const unsigned groups = (unsigned)std::min<uint64_t>(kFinalizeGroups, t.cpr);
    void* args[] = { &fa };
    const void* fn = t.acc_elem == 8 ? (const void*)&trace_finalize_kernel<double> : (const void*)&trace_finalize_kernel<float>;
    cudaError_t e = cudaLaunchKernel(fn, dim3(t.p.nfft / kFinalizeBins, (unsigned)nr), dim3(kFinalizeBins, groups), args, 0, stream);
    if (e != cudaSuccess) return cuda_fail(e, "launch trace_finalize_kernel");
    eng->launches++;
    return SA_OK;
}

int trace_device(Engine* eng, const void* d_iq, uint64_t n_samples, const TracePlan& t, void* const outs[3],
                 cudaStream_t stream) {
    const sa_spectrogram_params& p = t.p;
    int rc = eng->ensure_scratch(10, t.rows_per_group * t.cell_bytes() * t.nstats);
    if (rc) return rc;
    TraceCells tc;
    group_cells(eng, t, tc);
    for (uint64_t g0 = 0; g0 < t.n_rows; g0 += t.rows_per_group) {
        const uint64_t nr = std::min<uint64_t>(t.rows_per_group, t.n_rows - g0);
        const uint64_t f0 = g0 * t.fpr, nf = std::min<uint64_t>(nr * t.fpr, p.n_frames - f0);
        cudaError_t e = cudaMemsetAsync(eng->scratch[10], 0, t.rows_per_group * t.cell_bytes() * t.nstats, stream);
        if (e != cudaSuccess) return cuda_fail(e, "clear trace accumulator");
        sa_spectrogram_params q = p;
        q.start_sample = p.start_sample + f0 * p.hop;
        q.n_frames = nf;
        rc = eng->launch_spectrogram(d_iq, n_samples, q, t.prec, nullptr, stream, 2, POOL_TRACE, t.fpr, &tc);
        if (rc) return rc;
        rc = launch_finalize(eng, t, tc, nf, nr, outs, g0, stream);
        if (rc) return rc;
    }
    return SA_OK;
}

// Host buffer: per group of rows, chunks of frames stream through the three pipeline slots (H2D -> pooled transform on
// the slot's stream) into one accumulator; after the slots drain, one finalize, and only the rows cross PCIe.
int trace_host(Engine* eng, const void* iq, uint64_t iq_bytes, const TracePlan& t, void* const outs[3]) {
    const sa_spectrogram_params& p = t.p;
    const uint64_t bps = spec_bytes_per_iq(p);
    const uint64_t n_samples = iq_bytes / bps;
    // chunks bounded as the canvas path bounds them: the larger of the frames' dB rows and their input samples
    const uint64_t per_frame = std::max<uint64_t>((uint64_t)p.nfft * 4, p.hop * bps);
    const uint64_t fpc = std::min<uint64_t>(std::max<uint64_t>(1, eng->chunk_bytes / per_frame), p.n_frames);
    const uint64_t readable = n_samples > p.start_sample ? n_samples - p.start_sample : 0;
    const uint64_t in_cap = std::max<uint64_t>(16, std::min<uint64_t>((fpc - 1) * p.hop + p.nfft, readable) * bps);
    const uint64_t rows_bytes = t.rows_per_group * p.nfft * t.out_elem;
    int rc = eng->ensure_scratch(10, t.rows_per_group * t.cell_bytes() * t.nstats);
    if (rc == SA_OK) rc = eng->ensure_scratch(11, rows_bytes * t.nstats);
    if (rc) return rc;
    const bool in_pinned = host_ptr_is_pinned(iq);
    for (int i = 0; i < kSlots && rc == SA_OK; i++) {
        rc = eng->ensure_slot(eng->slots[i], in_cap, 0);
        if (rc == SA_OK) rc = eng->ensure_staging(eng->slots[i], in_pinned ? 0 : in_cap, 0);
    }
    if (rc) return rc;
    auto drain = [&](int rc0) {             // nothing may be in flight on the staging buffers or the caller's memory
        for (int i = 0; i < kSlots; i++) {
            cudaError_t e = cudaStreamSynchronize(eng->slots[i].stream);
            if (e != cudaSuccess && rc0 == SA_OK) rc0 = cuda_fail(e, "trace pipeline drain");
        }
        return rc0;
    };
    TraceCells tc;
    group_cells(eng, t, tc);
    void* d_rows[3] = {};
    for (int s = 0; s < 3; s++)
        if (outs[s]) d_rows[s] = (char*)eng->scratch[11] + t.stat_of[s] * rows_bytes;
    cudaStream_t s0 = eng->slots[0].stream;
    uint64_t c = 0;
    for (uint64_t g0 = 0; g0 < t.n_rows && rc == SA_OK; g0 += t.rows_per_group) {
        const uint64_t nr = std::min<uint64_t>(t.rows_per_group, t.n_rows - g0);
        const uint64_t gf0 = g0 * t.fpr, gnf = std::min<uint64_t>(nr * t.fpr, p.n_frames - gf0);
        // every slot has drained (the previous group's finalize read the cells): clear them before any chunk reduces
        cudaError_t e = cudaMemsetAsync(eng->scratch[10], 0, t.rows_per_group * t.cell_bytes() * t.nstats, s0);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s0);
        if (e != cudaSuccess) { rc = cuda_fail(e, "clear trace accumulator"); break; }
        for (uint64_t cf = 0; cf < gnf && rc == SA_OK; cf += fpc, c++) {
            Slot& s = eng->slots[c % kSlots];
            e = cudaStreamSynchronize(s.stream);              // slot buffers free again
            if (e != cudaSuccess) { rc = cuda_fail(e, "slot sync"); break; }
            const uint64_t nf = std::min<uint64_t>(fpc, gnf - cf);
            const uint64_t s_begin = p.start_sample + (gf0 + cf) * p.hop;
            uint64_t s_end = s_begin + (nf - 1) * p.hop + p.nfft;
            if (s_end > n_samples) s_end = n_samples;          // frames past EOF reduce the EOF power
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
            TraceCells tcc = tc;
            tcc.frame0 = cf;
            rc = eng->launch_spectrogram(s.d_in, ns, q, t.prec, nullptr, s.stream, 5 + (int)(c % kSlots), POOL_TRACE, t.fpr, &tcc);
        }
        rc = drain(rc);
        if (rc) break;
        rc = launch_finalize(eng, t, tc, gnf, nr, d_rows, 0, s0);
        for (int st = 0; st < 3 && rc == SA_OK; st++) {
            if (!outs[st]) continue;
            e = cudaMemcpyAsync((char*)outs[st] + g0 * p.nfft * t.out_elem, d_rows[st], nr * p.nfft * t.out_elem,
                                cudaMemcpyDeviceToHost, s0);
            if (e != cudaSuccess) rc = cuda_fail(e, "D2H trace rows");
        }
        cudaError_t e2 = cudaStreamSynchronize(s0);
        if (e2 != cudaSuccess && rc == SA_OK) rc = cuda_fail(e2, "trace rows");
    }
    return drain(rc);
}

}  // namespace

extern "C" {

int32_t sa_spectrum_trace(sa_engine* engine, const void* iq, uint64_t iq_bytes, const sa_spectrogram_params* params,
                          uint64_t frames_per_row, void* out_mean, void* out_max, void* out_min, uint64_t out_bytes) {
    ENGINE_ENTER(engine);
    void* outs[3] = { out_mean, out_max, out_min };
    TracePlan t;
    int rc = plan_trace(params, frames_per_row, outs, out_bytes, t);
    if (rc) return rc;
    if (!iq && iq_bytes) return set_error(SA_ERR_INVALID_ARG, "NULL buffer");
    if (strict_zero(t.p)) {                 // nothing is transformed: constant rows from the frame counts
        strict_trace_rows(t, iq_bytes / spec_bytes_per_iq(t.p), outs);
        engine->last_kernel = "none (strict_reference zero decode: constant trace rows)";
        return SA_OK;
    }
    return trace_host(engine, iq, iq_bytes, t, outs);
}

int32_t sa_spectrum_trace_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes, const sa_spectrogram_params* params,
                                 uint64_t frames_per_row, void* d_mean, void* d_max, void* d_min, uint64_t out_bytes,
                                 void* cuda_stream) {
    ENGINE_ENTER(engine);
    void* outs[3] = { d_mean, d_max, d_min };
    TracePlan t;
    int rc = plan_trace(params, frames_per_row, outs, out_bytes, t);
    if (rc) return rc;
    if (!d_iq && iq_bytes) return set_error(SA_ERR_INVALID_ARG, "NULL buffer");
    const uint64_t bps = spec_bytes_per_iq(t.p);
    if ((uintptr_t)d_iq % bps) return set_error(SA_ERR_INVALID_ARG, "d_iq must be aligned to %llu bytes", (unsigned long long)bps);
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (strict_zero(t.p)) {
        std::vector<char> h[3];
        void* hp[3] = {};
        const size_t bytes = t.n_rows * t.p.nfft * t.out_elem;
        for (int s = 0; s < 3; s++) if (outs[s]) { h[s].resize(bytes); hp[s] = h[s].data(); }
        strict_trace_rows(t, iq_bytes / bps, hp);
        for (int s = 0; s < 3; s++) {
            if (!outs[s]) continue;
            cudaError_t e = cudaMemcpyAsync(outs[s], hp[s], bytes, cudaMemcpyHostToDevice, stream);
            if (e != cudaSuccess) { cudaStreamSynchronize(stream); return cuda_fail(e, "H2D trace rows"); }
        }
        cudaError_t e = cudaStreamSynchronize(stream);           // the host rows go out of scope
        if (e != cudaSuccess) return cuda_fail(e, "H2D trace rows");
        engine->last_kernel = "none (strict_reference zero decode: constant trace rows)";
        return SA_OK;
    }
    return trace_device(engine, d_iq, iq_bytes / bps, t, outs, stream);
}

}  // extern "C"
