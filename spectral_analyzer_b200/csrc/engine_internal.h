// engine_internal.h -- host-side state behind the opaque sa_engine handle.
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <condition_variable>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/sa_engine.h"
#include "spectrogram_tma_kernel.cuh"
#include "spectrogram_mid_kernel.cuh"
#include "large_fft_kernels.cuh"

namespace sa {

int set_error(int code, const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
const SpecKernelInfo* find_spec_kernel(int prec, int n, int dk, int win, int tma);
const LargeKernelInfo* find_large_kernel(int prec, int n, int dk, int win);
void host_window(int window_id, int n, std::vector<double>& w);
int dtype_kind(int dtype);
bool host_ptr_is_pinned(const void* p);     // pinned / registered host memory (DMA-able as is)
int check_spec_params(const sa_spectrogram_params* p, int* prec_out);   // validates, resolves precision
void fill_load_params(LoadParams& lp, const void* base, int dtype, int big_endian);
uint64_t spec_bytes_per_iq(const sa_spectrogram_params& p);   // Global.getBytesPerSample, strict_reference aware
// strict_reference: datatypes SpectralService.computeMagnitudes has no branch for decode to zeros (:60-63)
inline bool strict_zero(const sa_spectrogram_params& p) {
    return p.strict_reference && (p.dtype == SA_CF64 || p.dtype == SA_DT_OTHER);
}

// Where the host pipeline takes a capture's bytes from: caller memory (pinned: DMA source as is; pageable:
// parallel memcpy into the pinned ring) or an open file (parallel pread straight into the pinned ring).
struct HostSource {
    const void* ptr = nullptr;
    int fd = -1;
    uint64_t file_off = 0;          // byte offset of sample 0 in the file (core:header_bytes, SigMfHelper.java:59-67)
};

// The engine's analysis profile: what JDSP decides inside Resampler.downConvert* / calculatePsdWelch
// (sa_analysis_config, include/sa_engine.h); defaults = the repository's documented spec.
struct AnalysisProfile {
    std::vector<double> taps;                 // empty: built-in Hamming-windowed sinc, 8*down+1 taps
    int delay_mode = SA_DELAY_CAUSAL;
    int length_mode = SA_LEN_FLOOR;
    int psd_scaling = SA_PSD_DENSITY;
    int psd_detrend = SA_DETREND_NONE;
    int psd_precision = SA_PREC_F32;
    int strict_reference = 0;
};

constexpr int kSlots = 3;
constexpr int kScratch = 14;

struct Slot {
    cudaStream_t stream = nullptr;
    void* d_in = nullptr;  size_t in_cap = 0;
    void* d_out = nullptr; size_t out_cap = 0;
    // pinned staging for PAGEABLE host buffers (an mmapped .sigmf-data file cannot be cudaHostRegister'ed)
    void* h_in = nullptr;  size_t h_in_cap = 0;
    void* h_out = nullptr; size_t h_out_cap = 0;
    void* pending_dst = nullptr; size_t pending_bytes = 0;       // result still sitting in h_out
};

// Worker threads that move bytes between pageable memory and the pinned staging buffers in parallel
// (one memcpy thread moves 5-10 GB/s; PCIe 5 x16 needs ~50 GB/s per direction).
class CopyPool {
public:
    explicit CopyPool(int workers);
    ~CopyPool();
    struct Group { size_t outstanding = 0; };                    // one asynchronous copy (start / wait)
    void copy(void* dst, const void* src, size_t bytes);         // returns when every part has been copied
    // same, the source being bytes [off, off + bytes) of an open file (parallel pread); false on a short read / error
    bool read(void* dst, int fd, uint64_t off, size_t bytes);
    // asynchronous memcpy: every part goes to the workers, the caller carries on (e.g. with the next chunk's copy-in) and
    // waits later; `g` must stay alive until wait() returns
    void start(void* dst, const void* src, size_t bytes, Group* g);
    void wait(Group* g);
private:
    void worker();
    void run(void* dst, const void* src, int fd, uint64_t off, size_t bytes);
    struct Job { char* dst; const char* src; size_t bytes; int fd; uint64_t off; Group* group; };
    std::atomic<bool> io_error_{false};
    std::vector<std::thread> threads_;
    std::mutex mu_;
    std::condition_variable cv_, done_cv_;
    std::vector<Job> queue_;
    bool stop_ = false;
};

struct Engine {
    int device = 0;
    int num_sms = 0;
    std::mutex mu;
    uint64_t launches = 0;
    std::string last_kernel;                         // name of the spectrogram kernel the last launch selected
    uint64_t chunk_bytes = 64ull << 20;              // per-slot staging size of the host pipeline
    std::map<uint64_t, void*> twiddles;              // (prec, nfft) -> device table
    std::map<uint64_t, void*> windows;               // (prec, window, nfft) -> device table
    std::map<uint64_t, void*> misc_tables;           // FIR taps etc.
    std::map<const void*, int> occupancy;            // kernel -> resident CTAs per SM
    std::vector<const void*> registered;             // cudaHostRegister'ed ranges
    Slot slots[kSlots];
    CopyPool* copy_pool = nullptr;                   // created on first use
    // device workspaces: [0] annotation plan + taps, [1] Welch plan + partial spectra, [2] four-step FFT,
    // [3] canvas / canvas dB rows, [4] signal lists of the packer / series kernels,
    // [5..7] four-step FFT workspaces of the host pipeline's slots (their chunks run concurrently on three streams)
    // [8..11] second four-step workspace of the same callers (two-stream chunk overlap, launch_spectrogram_large)
    // [12] FP32 rows the downconverter hands to the Welch kernels (two halves, reused batch after batch: L2 resident),
    // [13] Welch plan + partial spectra of the helper stream's batches
    void* scratch[kScratch] = {};
    size_t scratch_cap[kScratch] = {};
    cudaStream_t large_aux[4] = {};                  // helper stream per four-step caller (device API, slots 0..2)
    cudaEvent_t large_ev[4][2] = {};                 // fork / join events of that helper stream
    bool l2_persist_set = false; size_t l2_window_max = 0;   // persisting-L2 carve-out for the four-step workspace
    AnalysisProfile profile;                         // sa_set_analysis_config
    cudaStream_t dc_aux = nullptr;                   // annotation batches alternate between the caller's stream and this one
    cudaEvent_t dc_ev[2] = {};                       // fork / join
    cudaEvent_t dc_pipe_ev[4] = {};                  // pipelined batches: rows of batch parity p written [p], consumed [2 + p]
    int dc_aux_prio = 0;                             // 1: dc_aux was created as a high-priority stream
    void* h_plan = nullptr; size_t h_plan_cap = 0;   // pinned staging of a call's annotation / tap / Welch plans
    cudaEvent_t plan_ev = nullptr;                   // the last upload from h_plan has completed
    std::map<const void*, size_t> dc_smem_set;       // dynamic shared memory limit already granted per kernel

    ~Engine();
    int twiddle_table(const SpecKernelInfo& k, const void** d_tab);
    int window_table(int window_id, int n, int prec, const void** d_tab);
    int kernel_grid(const void* fn, int cta, size_t smem, int* blocks_per_sm);
    int ensure_slot(Slot& s, size_t in_bytes, size_t out_bytes);
    int ensure_staging(Slot& s, size_t in_bytes, size_t out_bytes);      // pinned h_in / h_out (0 = not needed)
    void host_copy(void* dst, const void* src, size_t bytes);            // parallel memcpy (CopyPool)
    bool host_read(void* dst, int fd, uint64_t off, size_t bytes);       // parallel pread (CopyPool)
    int flush_pending(Slot& s);                                          // h_out -> the caller's pageable buffer
    int ensure_scratch(int which, size_t bytes);
    int root_table(int n, int prec, const void** d_tab);      // W_n^j, j = 0..n-1
    int mid_t1_table(int n, const void** d_tab);              // pass-1 twiddle pairs of spectrogram_mid_kernel
    // ws: index of the scratch buffer the four-step path may use as its workspace (2 for device-API calls; the
    // host pipeline passes 5 + slot so that chunks in flight on different streams never share a workspace)
    int launch_spectrogram_large(const void* d_iq, uint64_t n_samples, const sa_spectrogram_params& p, int prec,
                                 const SpecArgs& base, void* d_out, cudaStream_t stream, int ws);
    // pool_mode != 0: instead of rows, |X|^2 is reduced (1 max, 2 sum) over the pool_fpc frames of each canvas column into
    // d_out = float[n_frames / pool_fpc][nfft], which the caller has zeroed (display.cu); transforms up to 16384 points.
    // A strict_zero request transforms nothing (its rows are constants): it takes the rows path, not the pooling one.
    int launch_spectrogram(const void* d_iq, uint64_t n_samples, const sa_spectrogram_params& p, int prec,
                           void* d_out, cudaStream_t stream, int ws = 2, int pool_mode = 0, uint64_t pool_fpc = 1);
    static bool can_pool(const sa_spectrogram_params& p, int prec) {
        return p.nfft <= 16384 && !(prec == SA_PREC_F64 && p.nfft > 8192) && !strict_zero(p);
    }
    int spectrogram_host(const HostSource& src, uint64_t iq_bytes, const sa_spectrogram_params& p, int prec, void* out);
};

}  // namespace sa

// The opaque handle of include/sa_engine.h.
struct sa_engine : public sa::Engine {};

// First statement of every entry point that takes an engine: NULL check, the per-engine lock (calls on one
// engine serialise; different engines run concurrently) and device selection for the calling thread.
#define ENGINE_ENTER(engine)                                                         \
    if (!(engine)) return set_error(SA_ERR_INVALID_ARG, "engine is NULL");            \
    std::lock_guard<std::mutex> lock_((engine)->mu);                                  \
    { cudaError_t e_ = cudaSetDevice((engine)->device);                               \
      if (e_ != cudaSuccess) return cuda_fail(e_, "cudaSetDevice"); }
