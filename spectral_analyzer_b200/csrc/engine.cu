// engine.cu -- C-ABI implementation (include/sa_engine.h): argument checking, plan/table cache,
// kernel selection, and the host<->device chunk pipeline.  No CPU fallback anywhere: every
// compute entry point launches CUDA kernels or fails.
#include "engine_internal.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cerrno>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

namespace sa {

#ifndef SA_LARGE_DUAL_DEFAULT
#define SA_LARGE_DUAL_DEFAULT 0
#endif
constexpr bool kLargeDualDefault = SA_LARGE_DUAL_DEFAULT != 0;
constexpr uint64_t kLargeDualWsMb = 48;

// ---------------- parallel host copies ----------------
CopyPool::CopyPool(int workers) {
    for (int i = 0; i < workers; i++) threads_.emplace_back([this] { worker(); });
}
CopyPool::~CopyPool() {
    { std::lock_guard<std::mutex> l(mu_); stop_ = true; }
    cv_.notify_all();
    for (auto& t : threads_) t.join();
}
void CopyPool::worker() {
    for (;;) {
        Job j;
        {
            std::unique_lock<std::mutex> l(mu_);
            cv_.wait(l, [this] { return stop_ || !queue_.empty(); });
            if (queue_.empty()) return;
            j = queue_.back();
            queue_.pop_back();
        }
        if (j.fd >= 0) {
            size_t done = 0;
            while (done < j.bytes) {
                const ssize_t r = pread(j.fd, j.dst + done, j.bytes - done, (off_t)(j.off + done));
                if (r <= 0) { io_error_ = true; break; }
                done += (size_t)r;
            }
        } else {
            memcpy(j.dst, j.src, j.bytes);
        }
        {
            std::lock_guard<std::mutex> l(mu_);
            if (--j.group->outstanding == 0) done_cv_.notify_all();
        }
    }
}
void CopyPool::run(void* dst, const void* src, int fd, uint64_t foff, size_t bytes) {
    const size_t part = std::max<size_t>(1 << 20, (bytes / (threads_.size() + 1) + 4095) & ~(size_t)4095);
    const size_t own_bytes = std::min(part, bytes);
    Group g;
    {
        std::lock_guard<std::mutex> l(mu_);
        for (size_t off = own_bytes; off < bytes; off += part) {
            queue_.push_back({(char*)dst + off, src ? (const char*)src + off : nullptr, std::min(part, bytes - off), fd, foff + off, &g});
            g.outstanding++;
        }
    }
    cv_.notify_all();
    if (fd >= 0) {                                    // the caller moves the first part
        size_t done = 0;
        while (done < own_bytes) {
            const ssize_t r = pread(fd, (char*)dst + done, own_bytes - done, (off_t)(foff + done));
            if (r <= 0) { io_error_ = true; break; }
            done += (size_t)r;
        }
    } else {
        memcpy(dst, src, own_bytes);
    }
    std::unique_lock<std::mutex> l(mu_);
    done_cv_.wait(l, [&g] { return g.outstanding == 0; });
}
void CopyPool::copy(void* dst, const void* src, size_t bytes) { run(dst, src, -1, 0, bytes); }
void CopyPool::start(void* dst, const void* src, size_t bytes, Group* g) {
    const size_t part = std::max<size_t>(1 << 20, (bytes / std::max<size_t>(1, threads_.size()) + 4095) & ~(size_t)4095);
    {
        std::lock_guard<std::mutex> l(mu_);
        for (size_t off = 0; off < bytes; off += part) {
            queue_.push_back({(char*)dst + off, (const char*)src + off, std::min(part, bytes - off), -1, 0, g});
            g->outstanding++;
        }
    }
    cv_.notify_all();
}
void CopyPool::wait(Group* g) {
    std::unique_lock<std::mutex> l(mu_);
    done_cv_.wait(l, [g] { return g->outstanding == 0; });
}
bool CopyPool::read(void* dst, int fd, uint64_t off, size_t bytes) {
    io_error_ = false;
    run(dst, nullptr, fd, off, bytes);
    return !io_error_;
}

bool host_ptr_is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
}

// ---------------- error reporting ----------------
static thread_local char g_err[512] = "";

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int cuda_fail(cudaError_t e, const char* what) {
    return set_error(e == cudaErrorMemoryAllocation ? SA_ERR_OOM : SA_ERR_CUDA, "%s: %s", what,
                     cudaGetErrorString(e));
}

// ---------------- kernel registry ----------------
static std::vector<SpecKernelInfo>& spec_registry() {
    static std::vector<SpecKernelInfo> r;
    return r;
}
void register_spec_kernel(const SpecKernelInfo& k) { spec_registry().push_back(k); }

const SpecKernelInfo* find_spec_kernel(int prec, int n, int dk, int win, int tma) {
    for (const auto& k : spec_registry())
        if (k.prec == prec && k.n == n && k.dk == dk && k.win == win && k.tma == tma) return &k;
    return nullptr;
}

static std::vector<LargeKernelInfo>& large_registry() {
    static std::vector<LargeKernelInfo> r;
    return r;
}
void register_large_kernel(const LargeKernelInfo& k) { large_registry().push_back(k); }
const LargeKernelInfo* find_large_kernel(int prec, int n, int dk, int win) {
    for (const auto& k : large_registry())
        if (k.prec == prec && k.n == n && k.dk == dk && k.win == win) return &k;
    return nullptr;
}

// ---------------- tables ----------------
void host_window(int window_id, int n, std::vector<double>& w) {
    w.resize(n);
    const double two_pi = 6.283185307179586476925286766559;
    for (int i = 0; i < n; i++) {
        const double x = two_pi * (double)i / (double)n;
        switch (window_id) {
            case SA_WIN_HANN:     w[i] = 0.5 - 0.5 * std::cos(x); break;
            case SA_WIN_HAMMING:  w[i] = 0.54 - 0.46 * std::cos(x); break;
            case SA_WIN_BLACKMAN: w[i] = 0.42 - 0.5 * std::cos(x) + 0.08 * std::cos(2 * x); break;
            case SA_WIN_BLACKMAN_HARRIS:
                w[i] = 0.35875 - 0.48829 * std::cos(x) + 0.14128 * std::cos(2 * x) - 0.01168 * std::cos(3 * x);
                break;
            default: w[i] = 1.0;
        }
    }
}

// Stockham twiddles in the order fft_pass reads them (fft_core.cuh): per pass, per sub-butterfly s,
// per m' < R/2, per thread t one PAIR (W for element m', W for element m' + R/2).
static void host_twiddles(int n, int p, int np, const int* radix, std::vector<double>& re, std::vector<double>& im) {
    const int tpf = n / p;
    re.assign((size_t)(np - 1) * n, 1.0);
    im.assign((size_t)(np - 1) * n, 0.0);
    const double two_pi = 6.283185307179586476925286766559;
    int ns = radix[0];
    for (int pass = 1; pass < np; pass++) {
        const int r = radix[pass], s_cnt = p / r;
        for (int s = 0; s < s_cnt; s++)
            for (int mp = 0; mp < r / 2; mp++)
                for (int t = 0; t < tpf; t++)
                    for (int h = 0; h < 2; h++) {
                        const int m = mp + h * (r / 2);
                        const int j = t + tpf * s;
                        const long long e = (long long)(j % ns) * m * (n / (ns * r));
                        const double ang = -two_pi * (double)(e % n) / (double)n;
                        const size_t idx = (size_t)(pass - 1) * n + ((size_t)(s * (r / 2) + mp) * tpf + t) * 2 + h;
                        re[idx] = std::cos(ang);
                        im[idx] = std::sin(ang);
                    }
        ns *= r;
    }
}

template <typename T>
static int upload_pairs(const std::vector<double>& re, const std::vector<double>& im, void** d_out) {
    std::vector<T> h(re.size() * 2);
    for (size_t i = 0; i < re.size(); i++) { h[2 * i] = (T)re[i]; h[2 * i + 1] = (T)im[i]; }
    cudaError_t e = cudaMalloc(d_out, h.size() * sizeof(T));
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(twiddle)");
    e = cudaMemcpy(*d_out, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
    // a pageable H2D cudaMemcpy may return once the data is STAGED; the kernels that read the table run on
    // non-blocking streams, which do not order against the legacy stream: wait for the DMA itself
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemcpy(twiddle)");
    return SA_OK;
}

int Engine::twiddle_table(const SpecKernelInfo& k, const void** d_tab) {
    // the table layout depends on the whole plan (p, passes, radices), not only on (precision, n)
    uint64_t plan = (uint64_t)k.p * 8 + (uint64_t)k.np;
    for (int i = 0; i < 4; i++) plan = plan * 131 + (uint64_t)k.radix[i];
    const uint64_t key = ((uint64_t)k.prec << 60) | ((plan & 0xFFFFFFFFFull) << 24) | (uint32_t)k.n;
    auto it = twiddles.find(key);
    if (it != twiddles.end()) { *d_tab = it->second; return SA_OK; }
    std::vector<double> re, im;
    host_twiddles(k.n, k.p, k.np, k.radix, re, im);
    void* d = nullptr;
    int rc = (k.prec == SA_PREC_F64) ? upload_pairs<double>(re, im, &d) : upload_pairs<float>(re, im, &d);
    if (rc) return rc;
    twiddles[key] = d;
    *d_tab = d;
    return SA_OK;
}

int Engine::window_table(int window_id, int n, int prec, const void** d_tab) {
    const uint64_t key = ((uint64_t)prec << 48) | ((uint64_t)window_id << 32) | (uint32_t)n;
    auto it = windows.find(key);
    if (it != windows.end()) { *d_tab = it->second; return SA_OK; }
    std::vector<double> w;
    host_window(window_id, n, w);
    void* d = nullptr;
    cudaError_t e;
    if (prec == SA_PREC_F64) {
        e = cudaMalloc(&d, n * sizeof(double));
        if (e == cudaSuccess) e = cudaMemcpy(d, w.data(), n * sizeof(double), cudaMemcpyHostToDevice);
    } else {
        std::vector<float> wf(w.begin(), w.end());
        e = cudaMalloc(&d, n * sizeof(float));
        if (e == cudaSuccess) e = cudaMemcpy(d, wf.data(), n * sizeof(float), cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();      // see upload_pairs
    if (e != cudaSuccess) return cuda_fail(e, "window table");
    windows[key] = d;
    *d_tab = d;
    return SA_OK;
}

int Engine::root_table(int n, int prec, const void** d_tab) {
    const uint64_t key = ((uint64_t)prec << 32) | (uint32_t)n;
    auto it = misc_tables.find(key);
    if (it != misc_tables.end()) { *d_tab = it->second; return SA_OK; }
    std::vector<double> re((size_t)n), im((size_t)n);
    const double two_pi = 6.283185307179586476925286766559;
    for (int j = 0; j < n; j++) { const double ang = -two_pi * (double)j / (double)n; re[j] = std::cos(ang); im[j] = std::sin(ang); }
    void* d = nullptr;
    int rc = (prec == SA_PREC_F64) ? upload_pairs<double>(re, im, &d) : upload_pairs<float>(re, im, &d);
    if (rc) return rc;
    misc_tables[key] = d;
    *d_tab = d;
    return SA_OK;
}

// Pass-1 twiddle pairs of spectrogram_mid_kernel: [m' < 16][r < R0] -> (W^(r m'), W^(r (m'+16))), W = W_{32 R0}
int Engine::mid_t1_table(int n, const void** d_tab) {
    const uint64_t key = (3ull << 40) | (uint32_t)n;
    auto it = misc_tables.find(key);
    if (it != misc_tables.end()) { *d_tab = it->second; return SA_OK; }
    const int r0 = n / 1024, len = 32 * r0;
    std::vector<double> re((size_t)32 * r0), im((size_t)32 * r0);
    const double two_pi = 6.283185307179586476925286766559;
    for (int mp = 0; mp < 16; mp++)
        for (int r = 0; r < r0; r++)
            for (int h = 0; h < 2; h++) {
                const int e = (r * (mp + 16 * h)) % len;
                const double ang = -two_pi * (double)e / (double)len;
                const size_t idx = ((size_t)mp * r0 + r) * 2 + h;
                re[idx] = std::cos(ang);
                im[idx] = std::sin(ang);
            }
    void* d = nullptr;
    int rc = upload_pairs<float>(re, im, &d);
    if (rc) return rc;
    misc_tables[key] = d;
    *d_tab = d;
    return SA_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point lookup (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            p = nullptr;
        }
        return (EncodeTiledFn)p;
    }();
    return fn;
}

// Four-step path (large_fft_kernels.cuh): frames are processed in chunks whose workspace stays L2-sized.
int Engine::launch_spectrogram_large(const void* d_iq, uint64_t n_samples, const sa_spectrogram_params& p, int prec,
                                     const SpecArgs& base, void* d_out, cudaStream_t stream, int ws) {
    (void)d_iq; (void)n_samples; (void)d_out;
    const int dk = dtype_kind(p.dtype);
    const int win = (prec == SA_PREC_F64) ? 1 : (p.window != SA_WIN_RECT ? 1 : 0);
    const LargeKernelInfo* k = find_large_kernel(prec, (int)p.nfft, dk, win);
    if (!k) return set_error(SA_ERR_UNSUPPORTED, "no kernel for nfft %u precision %s dtype %d", p.nfft,
                             prec == SA_PREC_F64 ? "f64" : "f32", p.dtype);
    LargeArgs a;
    memset(&a, 0, sizeof(a));
    a.s = base;
    // sub-transform tables come from the plans of the in-SM kernels of the same precision
    const SpecKernelInfo* k1 = find_spec_kernel(prec, k->n1, DK_CF32, 1, 0);
    const SpecKernelInfo* k2 = find_spec_kernel(prec, k->n2, DK_CF32, 1, 0);
    if (!k1 || !k2) return set_error(SA_ERR_UNSUPPORTED, "sub-transform plans %d / %d missing", k->n1, k->n2);
    int rc = twiddle_table(*k1, &a.s.twiddle);
    if (rc) return rc;
    rc = twiddle_table(*k2, &a.tw2);
    if (rc) return rc;
    rc = root_table((int)p.nfft, prec, &a.tw_n);
    if (rc) return rc;
    if (win) { rc = window_table(p.window, (int)p.nfft, prec, &a.s.window); if (rc) return rc; }
    const size_t elem = (prec == SA_PREC_F64) ? 16 : 8;
    const uint64_t per_frame = (uint64_t)p.nfft * elem;
    void* args[] = { &a };
    cudaError_t e;
    // 65536 points with 16-byte aligned frames, opt-in (SA_LARGE_ONCHIP=1): the on-chip cluster kernel (the frame stays
    // in the distributed shared memory of an 8-CTA cluster between the column and the row step; no workspace, DRAM
    // traffic = algorithmic bytes).  Measured on B200 it LOSES to the two-kernel path (config 5: 1.32 vs 0.785 ms; FP32:
    // 1.04 vs 0.683 ms): one 256-thread CTA per SM leaves every phase latency-bound and the phases of a frame are
    // serialised by two cluster barriers (per frame and CTA, FP64, cycles: column FFTs 11.3 k, barrier 2.1 k, DSMEM pull
    // 5.3 k = 24 B/clk, barrier 5.0 k, row FFTs 7.0 k, dB + store 8.9 k; TMA wait 0.8 k, i.e. the loads ARE hidden) --
    // the two kernels are issue-bound, not bound by the workspace round trip (DESIGN.md K6).
    const char* onchip_env = getenv("SA_LARGE_ONCHIP");               // read per call: the tests A/B the two paths
    const bool use_onchip = onchip_env ? atoi(onchip_env) != 0 : false;
    const uint64_t iq_b = (uint64_t)sa_bytes_per_iq(p.dtype);
    const bool aligned = ((uintptr_t)d_iq % 16 == 0) && ((p.start_sample * iq_b) % 16 == 0) && ((p.hop * iq_b) % 16 == 0);
    if (k->fn_cluster && use_onchip && aligned) {
        auto it = occupancy.find(k->fn_cluster);
        int n_clusters = 0;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = kLargeCluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.blockDim = dim3(k->cta_cluster);
        cfg.dynamicSmemBytes = k->smem_cluster;
        cfg.stream = stream;
        cfg.attrs = attr; cfg.numAttrs = 1;
        if (it == occupancy.end()) {
            e = cudaFuncSetAttribute(k->fn_cluster, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k->smem_cluster);
            if (e != cudaSuccess) return cuda_fail(e, "on-chip four-step smem attribute");
            cfg.gridDim = dim3(kLargeCluster * num_sms);
            e = cudaOccupancyMaxActiveClusters(&n_clusters, k->fn_cluster, &cfg);
            if (e != cudaSuccess || n_clusters < 1) { cudaGetLastError(); n_clusters = 0; }
            occupancy[k->fn_cluster] = n_clusters;
        } else {
            n_clusters = it->second;
        }
        // tensor map [frame][n1][n2] over the readable frames, in 8-byte elements: strides hop and 256 samples
        // (frames overlap when hop < nfft), box = 16 columns x 256 rows x 1 frame
        const uint64_t first_end = p.start_sample + p.nfft;
        const uint64_t n_read = n_samples >= first_end ? std::min<uint64_t>(p.n_frames, (n_samples - first_end) / p.hop + 1) : 0;
        CUtensorMap tmap;
        bool have_map = false;
        if (n_clusters > 0 && n_read > 0 && encode_tiled_fn()) {
            const cuuint64_t e8 = iq_b / 8;
            const cuuint64_t gdim[3] = { (cuuint64_t)k->n2 * e8, (cuuint64_t)k->n1, (cuuint64_t)n_read };
            const cuuint64_t gstr[2] = { (cuuint64_t)k->n2 * iq_b, (cuuint64_t)p.hop * iq_b };
            const cuuint32_t box[3] = { (cuuint32_t)(kLargeC * e8), (cuuint32_t)k->n1, 1 };
            const cuuint32_t estr[3] = { 1, 1, 1 };
            void* gaddr = (char*)const_cast<void*>(d_iq) + p.start_sample * iq_b;
            have_map = gstr[1] < (1ull << 40) &&
                       encode_tiled_fn()(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, gaddr, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                         CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
        }
        if (have_map) {
            const uint64_t use = std::min<uint64_t>((uint64_t)n_clusters, p.n_frames);
            a.ws = nullptr;
#if SA_ONCHIP_PROF
            rc = ensure_scratch(ws, (size_t)use * kLargeCluster * 16 * sizeof(long long));
            if (rc) return rc;
            a.ws = scratch[ws];
#endif
            a.frame0 = 0;
            cfg.gridDim = dim3((unsigned)(use * kLargeCluster));
            void* cargs[] = { &a, &tmap };
            e = cudaLaunchKernelExC(&cfg, k->fn_cluster, cargs);
            if (e != cudaSuccess) return cuda_fail(e, "launch large_onchip_kernel");
            launches++;
#if SA_ONCHIP_PROF
            if (getenv("SA_ONCHIP_PROF_DUMP")) {
                cudaStreamSynchronize(stream);
                std::vector<long long> h((size_t)use * kLargeCluster * 16);
                cudaMemcpy(h.data(), scratch[ws], h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
                double sum[16] = {0};
                for (size_t c = 0; c < (size_t)use * kLargeCluster; c++) for (int i = 0; i < 16; i++) sum[i] += (double)h[c * 16 + i];
                const double fr = (double)p.n_frames * kLargeCluster;       // CTA-frames
                fprintf(stderr, "onchip prof (cycles per frame, mean over CTAs):");
                for (int i = 0; i < 9; i++) fprintf(stderr, " p%d=%.0f", i, sum[i] / fr);
                fprintf(stderr, "\n");
            }
#endif
            static const char* const dkn[] = { "cf32", "ci16", "c8", "cf64" };
            char nm[160];
            snprintf(nm, sizeof(nm), "large_onchip_kernel<%s,%dx%d,%s,%s> (%d-CTA clusters x %d)", prec == SA_PREC_F64 ? "double" : "float",
                     k->n1, k->n2, dkn[dk], win ? "window" : "rect", kLargeCluster, n_clusters);
            last_kernel = nm;
            return SA_OK;
        }
    }
    // Fused persistent kernel, opt-in (SA_LARGE_FUSED=1): both steps in one launch, work items drawn from a ticket counter,
    // workspace = an L2-persisting ring of frames (DRAM traffic ~ the algorithmic bytes).  Measured on B200: config 5 0.84-0.86 ms
    // against 0.78 ms for the two kernels below, FP32 65536 1.08-1.30 against 0.69 ms (without the persisting window 1.25 /
    // 1.52 ms): the per-item device-wide fence, the ticket round trip and two CTAs per SM cost more than the saved
    // traffic buys (profiles/r02_c5_onchip_ablation.txt).
    {
        const char* fused_env = getenv("SA_LARGE_FUSED");
        const bool fused_on = fused_env ? atoi(fused_env) != 0 : false;
        const char* ring_env = getenv("SA_LARGE_RING");
        const char* delay_env = getenv("SA_LARGE_DELAY");
        if (k->fn_fused && fused_on) {
            int ring = ring_env ? atoi(ring_env) : (int)std::max<uint64_t>(24, (40ull << 20) / per_frame);
            int delay = delay_env ? atoi(delay_env) : 12;
            if (delay < 1) delay = 1;
            if (ring < delay + 12) ring = delay + 12;
            if (!l2_persist_set) {
                cudaDeviceProp prop;
                if (cudaGetDeviceProperties(&prop, device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
                    cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)prop.persistingL2CacheMaxSize);
                    l2_window_max = (size_t)prop.accessPolicyMaxWindowSize;
                }
                cudaGetLastError();
                l2_persist_set = true;
            }
            const size_t ring_bytes = ((size_t)ring * per_frame + 255) & ~(size_t)255;
            const size_t ctr_bytes = (16 + 2 * (size_t)p.n_frames * sizeof(int) + 255) & ~(size_t)255;
            rc = ensure_scratch(ws, ring_bytes + ctr_bytes);
            if (rc) return rc;
            char* base_ws = (char*)scratch[ws];
            e = cudaMemsetAsync(base_ws + ring_bytes, 0, ctr_bytes, stream);
            if (e != cudaSuccess) return cuda_fail(e, "clear four-step counters");
            LargeFusedArgs fa;
            memset(&fa, 0, sizeof(fa));
            fa.a = a;
            fa.a.ws = base_ws;
            fa.a.frame0 = 0;
            fa.ticket = (unsigned long long*)(base_ws + ring_bytes);
            fa.cols_done = (int*)(base_ws + ring_bytes + 16);
            fa.rows_done = fa.cols_done + p.n_frames;
            fa.ring = ring; fa.delay = delay;
            int bps_f = 0;
            rc = kernel_grid(k->fn_fused, k->cta_cols, k->smem_fused, &bps_f);
            if (rc) return rc;
            const long long n_items = ((long long)p.n_frames + delay) * (k->n2 / kLargeC + k->n1 / kLargeC);
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
            attr[0].val.accessPolicyWindow.base_ptr = base_ws;
            attr[0].val.accessPolicyWindow.num_bytes = std::min<size_t>(ring_bytes, l2_window_max);
            attr[0].val.accessPolicyWindow.hitRatio = 1.0f;
            attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.stream = stream;
            const char* pers_env = getenv("SA_LARGE_PERSIST");
            const bool pers = l2_window_max > 0 && !(pers_env && atoi(pers_env) == 0);
            cfg.attrs = attr; cfg.numAttrs = pers ? 1 : 0;
            cfg.gridDim = dim3((unsigned)std::min<long long>(n_items, (long long)bps_f * num_sms));
            cfg.blockDim = dim3(k->cta_cols);
            cfg.dynamicSmemBytes = k->smem_fused;
            void* fargs[] = { &fa };
            e = cudaLaunchKernelExC(&cfg, k->fn_fused, fargs);
            if (e != cudaSuccess) return cuda_fail(e, "launch large_fused_kernel");
            launches++;
            static const char* const dkn[] = { "cf32", "ci16", "c8", "cf64" };
            char nm[160];
            snprintf(nm, sizeof(nm), "large_fused_kernel<%s,%dx%d,%s,%s> (ring %d, delay %d)", prec == SA_PREC_F64 ? "double" : "float",
                     k->n1, k->n2, dkn[dk], win ? "window" : "rect", ring, delay);
            last_kernel = nm;
            return SA_OK;
        }
    }
    // Two workspaces, two streams: even chunks run on the caller's stream, odd chunks on a helper stream forked
    // from it, so that one chunk's column pass fills the SMs the other chunk's row pass leaves idle in its last
    // wave, and workspaces small enough to stay in L2 no longer mean under-filled grids (SA_LARGE_DUAL=0 disables).
    static const char* dual_env = getenv("SA_LARGE_DUAL");
    static const bool dual_on = dual_env ? atoi(dual_env) != 0 : kLargeDualDefault;
    // SA_LARGE_PERSIST=1: the workspace is declared L2-persisting for the two kernels (launch attribute access policy
    // window, hit ratio 1, everything else streaming), so that the column kernel's A[k1][n2] stays in L2 until the row
    // kernel has read it instead of making a DRAM round trip; needs a workspace well below the persisting carve-out
    static const char* persist_env = getenv("SA_LARGE_PERSIST");
    static const bool persist_on = persist_env ? atoi(persist_env) != 0 : false;
    static const uint64_t ws_mb = getenv("SA_LARGE_WS_MB") ? (uint64_t)atoi(getenv("SA_LARGE_WS_MB"))
                                                            : (persist_on ? 32 : (dual_on ? kLargeDualWsMb : 512));
    if (persist_on && !l2_persist_set) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess && prop.persistingL2CacheMaxSize > 0) {
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, (size_t)prop.persistingL2CacheMaxSize);
            l2_window_max = (size_t)prop.accessPolicyMaxWindowSize;
        }
        cudaGetLastError();
        l2_persist_set = true;
    }
    const uint64_t chunk = std::max<uint64_t>(1, std::min<uint64_t>(p.n_frames, (ws_mb << 20) / per_frame));
    const bool dual = dual_on && p.n_frames > chunk;
    const int ai = (ws == 2) ? 0 : ws - 4;                 // helper index: device API 0, host-pipeline slots 1..3
    rc = ensure_scratch(ws, chunk * per_frame);
    if (rc) return rc;
    if (dual) {
        rc = ensure_scratch(8 + ai, chunk * per_frame);
        if (rc) return rc;
        if (!large_aux[ai]) {
            e = cudaStreamCreateWithFlags(&large_aux[ai], cudaStreamNonBlocking);
            for (int j = 0; j < 2 && e == cudaSuccess; j++) e = cudaEventCreateWithFlags(&large_ev[ai][j], cudaEventDisableTiming);
            if (e != cudaSuccess) return cuda_fail(e, "four-step helper stream");
        }
        e = cudaEventRecord(large_ev[ai][0], stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(large_aux[ai], large_ev[ai][0], 0);
        if (e != cudaSuccess) return cuda_fail(e, "four-step fork");
    }
    e = cudaFuncSetAttribute(k->fn_cols, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k->smem_cols);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k->fn_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k->smem_rows);
    if (e != cudaSuccess) return cuda_fail(e, "large FFT smem attribute");
    uint64_t c = 0;
    for (uint64_t f0 = 0; f0 < p.n_frames; f0 += chunk, c++) {
        const unsigned nf = (unsigned)std::min<uint64_t>(chunk, p.n_frames - f0);
        const bool odd = dual && (c & 1);
        cudaStream_t st = odd ? large_aux[ai] : stream;
        a.ws = scratch[odd ? 8 + ai : ws];
        a.frame0 = (long long)f0;
        if (persist_on && l2_window_max > 0) {
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeAccessPolicyWindow;
            attr[0].val.accessPolicyWindow.base_ptr = a.ws;
            attr[0].val.accessPolicyWindow.num_bytes = std::min<size_t>((size_t)nf * per_frame, l2_window_max);
            attr[0].val.accessPolicyWindow.hitRatio = 1.0f;
            attr[0].val.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            attr[0].val.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.stream = st; cfg.attrs = attr; cfg.numAttrs = 1;
            cfg.gridDim = dim3(k->n2 / kLargeC, nf); cfg.blockDim = dim3(k->cta_cols); cfg.dynamicSmemBytes = k->smem_cols;
            e = cudaLaunchKernelExC(&cfg, k->fn_cols, args);
            if (e != cudaSuccess) return cuda_fail(e, "launch large_cols_kernel");
            cfg.gridDim = dim3(k->n1 / kLargeC, nf); cfg.blockDim = dim3(k->cta_rows); cfg.dynamicSmemBytes = k->smem_rows;
            e = cudaLaunchKernelExC(&cfg, k->fn_rows, args);
            if (e != cudaSuccess) return cuda_fail(e, "launch large_rows_kernel");
            launches += 2;
            continue;
        }
        e = cudaLaunchKernel(k->fn_cols, dim3(k->n2 / kLargeC, nf), dim3(k->cta_cols), args, k->smem_cols, st);
        if (e != cudaSuccess) return cuda_fail(e, "launch large_cols_kernel");
        e = cudaLaunchKernel(k->fn_rows, dim3(k->n1 / kLargeC, nf), dim3(k->cta_rows), args, k->smem_rows, st);
        if (e != cudaSuccess) return cuda_fail(e, "launch large_rows_kernel");
        launches += 2;
    }
    {
        static const char* const dkn[] = { "cf32", "ci16", "c8", "cf64" };
        char nm[160];
        snprintf(nm, sizeof(nm), "large_cols_kernel+large_rows_kernel<%s,%dx%d,%s,%s>", prec == SA_PREC_F64 ? "double" : "float",
                 k->n1, k->n2, dkn[dk], win ? "window" : "rect");
        last_kernel = nm;
    }
    if (dual) {
        e = cudaEventRecord(large_ev[ai][1], large_aux[ai]);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, large_ev[ai][1], 0);
        if (e != cudaSuccess) return cuda_fail(e, "four-step join");
    }
    return SA_OK;
}

int Engine::kernel_grid(const void* fn, int cta, size_t smem, int* blocks_per_sm) {
    auto it = occupancy.find(fn);
    if (it != occupancy.end()) { *blocks_per_sm = it->second; return SA_OK; }
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(smem)");
    int nb = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, fn, cta, smem);
    if (e != cudaSuccess) return cuda_fail(e, "occupancy query");
    if (nb < 1) return set_error(SA_ERR_CUDA, "kernel does not fit on an SM (smem %zu)", smem);
    occupancy[fn] = nb;
    *blocks_per_sm = nb;
    return SA_OK;
}

int dtype_kind(int dtype) {
    switch (dtype) {
        case SA_CF32: return DK_CF32;
        case SA_CI16: return DK_CI16;
        case SA_CU8:
        case SA_CI8:  return DK_C8;
        case SA_CF64: return DK_CF64;
        default:      return -1;
    }
}

void fill_load_params(LoadParams& lp, const void* base, int dtype, int big_endian) {
    lp.base = base;
    lp.swap = big_endian ? 1 : 0;
    lp.c8_flip = (dtype == SA_CI8) ? 0x80808080u : 0u;
    lp.c8_off = (dtype == SA_CI8) ? 1.0f : 127.5f / 128.0f;
    lp.c8_c = 256.0f + lp.c8_off;
}

static bool is_pow2(uint64_t x) { return x && !(x & (x - 1)); }

// bytes per IQ pair as the frame loop sees them: Global.getBytesPerSample (S/sigmf/Global.java:67-79), fallback 8
uint64_t spec_bytes_per_iq(const sa_spectrogram_params& p) {
    if (p.dtype == SA_DT_OTHER) return p.strict_reference ? 8 : 0;
    return (uint64_t)sa_bytes_per_iq(p.dtype);
}

// rows of a strict_zero request: every readable frame is 20 log10(0 + 1e-10) = -200 dB (10 log10(1e-20) in power
// mode), frames past the end are eof_fill
__global__ void strict_fill_kernel(const SpecArgs a, const int nfft) {
    const long long frame = blockIdx.x;
    const bool readable = a.start_sample + frame * a.hop + nfft <= a.n_samples;      // MainController.java:987
    const double v = readable ? -200.0 : a.eof_fill;
    const size_t row = (size_t)frame * nfft;
    for (int k = threadIdx.x; k < nfft; k += blockDim.x) {
        if (a.out_kind == OUT_F32_DB) reinterpret_cast<float*>(a.out)[row + k] = (float)v;
        else if (a.out_kind == OUT_F64_DB) reinterpret_cast<double*>(a.out)[row + k] = v;
        else reinterpret_cast<uint32_t*>(a.out)[row + k] = colormap_rgba((float)v, a);
    }
}

static size_t out_elem_bytes(int out_kind) { return out_kind == SA_OUT_F64_DB ? 8 : 4; }

// Validates a request and resolves precision; returns SA_OK or an error.
int check_spec_params(const sa_spectrogram_params* p, int* prec_out) {
    if (!p) return set_error(SA_ERR_INVALID_ARG, "params is NULL");
    if (p->struct_size != sizeof(sa_spectrogram_params))
        return set_error(SA_ERR_INVALID_ARG, "params.struct_size %u != %zu", p->struct_size, sizeof(sa_spectrogram_params));
    if (p->dtype == SA_DT_OTHER && !p->strict_reference)
        return set_error(SA_ERR_UNSUPPORTED, "datatype without a decode branch (SA_DT_OTHER) needs strict_reference");
    if (spec_bytes_per_iq(*p) == 0) return set_error(SA_ERR_INVALID_ARG, "unknown dtype %d", p->dtype);
    if (!is_pow2(p->nfft))   // commons-math3 throws MathIllegalArgumentException (SpectralService.java:29)
        return set_error(SA_ERR_INVALID_ARG, "nfft %u is not a power of two", p->nfft);
    if (p->nfft < 64 || p->nfft > 65536)
        return set_error(SA_ERR_UNSUPPORTED, "nfft %u outside 64..65536 (main-scene.fxml:129)", p->nfft);
    if (p->hop == 0) return set_error(SA_ERR_INVALID_ARG, "hop is 0");
    // frame starts and output offsets are 64-bit signed on the device (MainController.java:984 extended to int64)
    const uint64_t lim = 1ull << 62;
    if (p->start_sample >= lim || p->hop >= lim || (p->n_frames && p->hop > (lim - p->start_sample) / p->n_frames))
        return set_error(SA_ERR_INVALID_ARG, "start_sample + n_frames * hop overflows 62 bits");
    if (p->n_frames > lim / ((uint64_t)p->nfft * 8))
        return set_error(SA_ERR_INVALID_ARG, "n_frames * nfft output bytes overflow 62 bits");
    if (p->window < SA_WIN_RECT || p->window > SA_WIN_BLACKMAN_HARRIS) return set_error(SA_ERR_INVALID_ARG, "unknown window %d", p->window);
    if (p->db_mode != SA_DB_MAG_1E10 && p->db_mode != SA_DB_POWER) return set_error(SA_ERR_INVALID_ARG, "unknown db_mode %d", p->db_mode);
    if (p->out_kind < SA_OUT_F32_DB || p->out_kind > SA_OUT_RGBA8) return set_error(SA_ERR_INVALID_ARG, "unknown out_kind %d", p->out_kind);
    if (p->out_kind == SA_OUT_RGBA8) {
        if (!(p->sample_rate > 0.0)) return set_error(SA_ERR_INVALID_ARG, "RGBA8 output needs sample_rate > 0");
        if (!(p->max_db > p->min_db)) return set_error(SA_ERR_INVALID_ARG, "RGBA8 output needs max_db > min_db");
        if (p->colormap != SA_CMAP_GRAYSCALE && p->colormap != SA_CMAP_HEATMAP) return set_error(SA_ERR_INVALID_ARG, "unknown colormap %d", p->colormap);
    }
    int prec = p->precision;
    if (prec == SA_PREC_AUTO) prec = (p->dtype == SA_CF64) ? SA_PREC_F64 : SA_PREC_F32;
    if (prec != SA_PREC_F32 && prec != SA_PREC_F64) return set_error(SA_ERR_INVALID_ARG, "unknown precision %d", p->precision);
    if (p->dtype == SA_CF64 && prec == SA_PREC_F32 && !p->strict_reference)
        return set_error(SA_ERR_UNSUPPORTED, "cf64 input runs on the FP64 path only");
    *prec_out = prec;
    return SA_OK;
}

// Launches the fused spectrogram kernel on device-resident samples.
int Engine::launch_spectrogram(const void* d_iq, uint64_t n_samples, const sa_spectrogram_params& p, int prec,
                               void* d_out, cudaStream_t stream, int ws, int pool_mode, uint64_t pool_fpc) {
    if (p.n_frames == 0) return SA_OK;
    const int dk = dtype_kind(p.dtype);
    const int win = (prec == SA_PREC_F64) ? 1 : (p.window != SA_WIN_RECT ? 1 : 0);
    SpecArgs a;
    memset(&a, 0, sizeof(a));
    fill_load_params(a.lp, d_iq, p.dtype, p.big_endian);
    a.n_samples = (long long)n_samples;
    a.start_sample = (long long)p.start_sample;
    a.hop = (long long)p.hop;
    a.n_frames = (long long)p.n_frames;
    a.out = d_out;
    a.out_kind = p.out_kind;
    a.db_mode = p.db_mode;
    a.eof_fill = p.eof_fill_db;
    if (p.out_kind == SA_OUT_RGBA8) {
        const double conv = 10.0 * std::log10(p.sample_rate / (double)p.nfft) + 20.0 * std::log10((double)p.nfft);
        a.inv_range = (float)(1.0 / (p.max_db - p.min_db));
        a.cmap_bias = (float)(-(conv + p.min_db) / (p.max_db - p.min_db));
        a.cmap = p.colormap;
    }
    if (pool_mode) {
        if (!can_pool(p, prec)) return set_error(SA_ERR_UNSUPPORTED, "fused pooling covers the in-SM transforms only");
        a.pool_mode = pool_mode;
        a.pool_fpc = (long long)std::max<uint64_t>(1, pool_fpc);
        a.pool_magic = a.pool_fpc > 1 ? (unsigned long long)((((unsigned __int128)1 << 64) + (unsigned __int128)(a.pool_fpc - 1)) / (unsigned __int128)a.pool_fpc) : 0ull;
        // |X|^2 whose level equals eof_fill_db: (10^(dB/20) - 1e-10)^2, or 10^(dB/10) - 1e-20 in power mode
        const double lin = p.db_mode == SA_DB_MAG_1E10 ? std::max(0.0, std::pow(10.0, p.eof_fill_db / 20.0) - 1e-10)
                                                       : 0.0;
        a.pool_eof = (float)(p.db_mode == SA_DB_MAG_1E10 ? lin * lin : std::max(0.0, std::pow(10.0, p.eof_fill_db / 10.0) - 1e-20));
    }
    if (strict_zero(p)) {                  // no sample is ever read
        for (uint64_t f0 = 0; f0 < p.n_frames; f0 += 65535u * 1024u) {
            const unsigned nf = (unsigned)std::min<uint64_t>(p.n_frames - f0, 65535u * 1024u);
            SpecArgs b = a;
            b.start_sample = a.start_sample + (long long)(f0 * p.hop);
            b.out = (char*)d_out + f0 * p.nfft * out_elem_bytes(p.out_kind);
            int n = (int)p.nfft;
            void* fargs[] = { &b, &n };
            cudaError_t fe = cudaLaunchKernel((const void*)&strict_fill_kernel, dim3(nf), dim3(256), fargs, 0, stream);
            if (fe != cudaSuccess) return cuda_fail(fe, "launch strict_fill_kernel");
            launches++;
        }
        last_kernel = "strict_fill_kernel";
        return SA_OK;
    }
    // transforms too large for one SM's shared memory take the four-step path
    if (p.nfft > 16384 || (prec == SA_PREC_F64 && p.nfft > 8192))
        return launch_spectrogram_large(d_iq, n_samples, p, prec, a, d_out, stream, ws);
    // TMA-staged variant (needs every frame start 16-byte aligned), else the LDG kernel
    const uint64_t iq_b = (uint64_t)sa_bytes_per_iq(p.dtype);
    const bool aligned = ((uintptr_t)d_iq % 16 == 0) && ((p.start_sample * iq_b) % 16 == 0) && ((p.hop * iq_b) % 16 == 0);
    static const bool no_tma = getenv("SA_NO_TMA") != nullptr;      // A/B switches for the ablations in DESIGN.md
    static const bool no_mid = getenv("SA_NO_MID") != nullptr;
    const SpecKernelInfo* k = (aligned && !no_tma) ? find_spec_kernel(prec, (int)p.nfft, dk, win, 1) : nullptr;
    // 4096: two radix-64 passes (one exchange) for cf32 / ci16 input; cu8 / ci8 keep the 3-pass kernel (measured)
    static const char* r64_env = getenv("SA_R64");
    const bool use_r64 = r64_env ? (strcmp(r64_env, "all") == 0) : (dk == DK_CF32 || dk == DK_CI16);
    // (the radix-64 kernel has its own store code: pooled launches take the small-radix-first kernel)
    if (!k && aligned && use_r64 && !pool_mode && prec == SA_PREC_F32 && p.nfft == 4096) k = find_spec_kernel(prec, 4096, dk, win, 4);
    // 2048: two warp-private 1024-point transforms + a radix-2 combine.  Opt-in (SA_SPLIT=1): measured against the
    // three-pass kernel on cu8 input it executes the same 43.8 instructions per point with 29 % fewer shared-memory
    // wavefronts and runs 2.02 vs 2.00 ms per 2^30 samples (f32 dB), 4.81 vs 4.51 ms per 2^31 (RGBA): both kernels
    // wait on the FMA pipe, not on shared memory
    const char* split_env = getenv("SA_SPLIT");
    const bool use_split = split_env ? atoi(split_env) != 0 : false;
    if (!k && aligned && use_split && !pool_mode && prec == SA_PREC_F32 && p.nfft == 2048) k = find_spec_kernel(prec, 2048, dk, win, 5);
    if (!k && aligned && !no_mid) {                                                        // small-radix-first plan
        // the asynchronously staged variant where it measured faster on B200 (tools/mid_pf_matrix.py): 2048 (8 frames
        // per CTA) and 16384 (one frame owns the SM) gain 6-19 %, 4096 (4 frames per CTA) 0-10 %, 8192 loses up to 19 %.
        // SA_MID_PF=all|none overrides.
        static const char* pf_env = getenv("SA_MID_PF");
        const bool pf = pf_env ? (strcmp(pf_env, "all") == 0) : (p.nfft != 8192);
        if (pf) k = find_spec_kernel(prec, (int)p.nfft, dk, win, 3);
        if (!k) k = find_spec_kernel(prec, (int)p.nfft, dk, win, 2);
    }
    if (!k) k = find_spec_kernel(prec, (int)p.nfft, dk, win, 0);
    if (!k) return set_error(SA_ERR_UNSUPPORTED, "no kernel for nfft %u precision %s dtype %d", p.nfft,
                             prec == SA_PREC_F64 ? "f64" : "f32", p.dtype);
    int rc;
    if (k->tma >= 2) {
        rc = mid_t1_table(k->n, &a.twiddle);
        if (rc) return rc;
        rc = root_table(k->n, prec, &a.aux);
    } else {
        rc = twiddle_table(*k, &a.twiddle);
    }
    if (rc) return rc;
    if (win) { rc = window_table(p.window, (int)p.nfft, prec, &a.window); if (rc) return rc; }
    int bps = 0;
    rc = kernel_grid(k->fn, k->cta, k->smem, &bps);
    if (rc) return rc;
    const long long n_blocks = ((long long)p.n_frames + k->fpc - 1) / k->fpc;
    const long long max_grid = (long long)bps * num_sms;
    const unsigned grid = (unsigned)std::min<long long>(n_blocks, max_grid);
    void* args[] = { &a };
    cudaError_t e = cudaLaunchKernel(k->fn, dim3(grid), dim3(k->cta), args, k->smem, stream);
    if (e != cudaSuccess) return cuda_fail(e, "launch spectrogram_kernel");
    launches++;
    {
        static const char* const fam[] = { "spectrogram_kernel", "spectrogram_tma_kernel", "spectrogram_mid_kernel",
                                           "spectrogram_mid_kernel(prefetch)", "spectrogram_r64_kernel", "spectrogram_split_kernel" };
        static const char* const dkn[] = { "cf32", "ci16", "c8", "cf64" };
        char nm[128];
        snprintf(nm, sizeof(nm), "%s<%s,%d,%s,%s>", fam[k->tma], prec == SA_PREC_F64 ? "double" : "float", k->n, dkn[k->dk],
                 k->win ? "window" : "rect");
        last_kernel = nm;
    }
    return SA_OK;
}

static CopyPool* make_copy_pool() {
    const char* ev = getenv("SA_COPY_THREADS");
    const unsigned hw = std::thread::hardware_concurrency();
    // all cores, at most 32: measured on the 16-vCPU B200 hosts (2 GiB mapped file in, pageable out): 8 / 11 / 16 / 24 threads =
    // 137 / 115 / 102 / 113 ms
    int n = ev ? atoi(ev) : (int)std::min(32u, std::max(2u, hw));
    return new CopyPool(std::max(1, n - 1));
}

void Engine::host_copy(void* dst, const void* src, size_t bytes) {
    if (bytes < (4u << 20)) { memcpy(dst, src, bytes); return; }
    if (!copy_pool) copy_pool = make_copy_pool();
    copy_pool->copy(dst, src, bytes);
}

bool Engine::host_read(void* dst, int fd, uint64_t off, size_t bytes) {
    if (!copy_pool) copy_pool = make_copy_pool();
    return copy_pool->read(dst, fd, off, bytes);
}

int Engine::ensure_staging(Slot& s, size_t in_bytes, size_t out_bytes) {
    cudaError_t e;
    if (s.h_in_cap < in_bytes) {
        if (s.h_in) cudaFreeHost(s.h_in);
        s.h_in = nullptr; s.h_in_cap = 0;
        e = cudaHostAlloc(&s.h_in, in_bytes, cudaHostAllocPortable);
        if (e != cudaSuccess) return cuda_fail(e, "cudaHostAlloc(staging in)");
        s.h_in_cap = in_bytes;
    }
    if (s.h_out_cap < out_bytes) {
        if (s.h_out) cudaFreeHost(s.h_out);
        s.h_out = nullptr; s.h_out_cap = 0;
        e = cudaHostAlloc(&s.h_out, out_bytes, cudaHostAllocPortable);
        if (e != cudaSuccess) return cuda_fail(e, "cudaHostAlloc(staging out)");
        s.h_out_cap = out_bytes;
    }
    return SA_OK;
}

int Engine::flush_pending(Slot& s) {
    if (!s.pending_dst) return SA_OK;
    host_copy(s.pending_dst, s.h_out, s.pending_bytes);
    s.pending_dst = nullptr; s.pending_bytes = 0;
    return SA_OK;
}

int Engine::ensure_slot(Slot& s, size_t in_bytes, size_t out_bytes) {
    cudaError_t e;
    if (!s.stream) {
        e = cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) return cuda_fail(e, "cudaStreamCreate");
    }
    if (s.in_cap < in_bytes) {
        if (s.d_in) cudaFree(s.d_in);
        s.d_in = nullptr; s.in_cap = 0;
        e = cudaMalloc(&s.d_in, in_bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(chunk in)");
        s.in_cap = in_bytes;
    }
    if (s.out_cap < out_bytes) {
        if (s.d_out) cudaFree(s.d_out);
        s.d_out = nullptr; s.out_cap = 0;
        e = cudaMalloc(&s.d_out, out_bytes);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(chunk out)");
        s.out_cap = out_bytes;
    }
    return SA_OK;
}

// Host-buffer spectrogram: frames are cut into chunks; chunk c runs H2D -> kernel -> D2H on
// slot c % kSlots' stream, so copies of one chunk overlap the kernel of another.
int Engine::spectrogram_host(const HostSource& hs, uint64_t iq_bytes, const sa_spectrogram_params& p, int prec, void* out) {
    const void* iq = hs.ptr;
    const uint64_t bps = spec_bytes_per_iq(p);
    const bool no_data = strict_zero(p);
    const uint64_t n_samples = iq_bytes / bps;
    const uint64_t obytes = out_elem_bytes(p.out_kind);
    const uint64_t row_bytes = (uint64_t)p.nfft * obytes;
    // frames per chunk: bound the larger of the two buffers by chunk_bytes
    const uint64_t per_frame = std::max<uint64_t>(p.hop * bps, row_bytes);
    uint64_t fpc = std::max<uint64_t>(1, chunk_bytes / per_frame);
    fpc = std::min<uint64_t>(fpc, p.n_frames);
    const uint64_t in_cap = ((fpc - 1) * p.hop + p.nfft) * bps;
    const uint64_t out_cap = fpc * row_bytes;
    // pageable buffers (an mmapped file, a Java heap array) go through pinned staging with parallel host copies;
    // pinned / registered buffers are the DMA source and target themselves
    const bool in_pinned = hs.fd < 0 && host_ptr_is_pinned(iq), out_pinned = host_ptr_is_pinned(out);
    int rc = SA_OK;
    uint64_t c = 0;
    for (uint64_t f0 = 0; f0 < p.n_frames && rc == SA_OK; f0 += fpc, c++) {
        Slot& s = slots[c % kSlots];
        rc = ensure_slot(s, in_cap, out_cap);
        if (rc) break;
        rc = ensure_staging(s, in_pinned ? 0 : in_cap, out_pinned ? 0 : out_cap);
        if (rc) break;
        cudaError_t e = cudaStreamSynchronize(s.stream);     // slot buffers free again
        if (e != cudaSuccess) { rc = cuda_fail(e, "slot sync"); break; }
        // the slot's previous result leaves its pinned buffer on the pool WHILE this chunk's samples are copied in
        CopyPool::Group drain;
        struct DrainGuard {                                  // the group must outlive its jobs on every exit path
            CopyPool* pool = nullptr; CopyPool::Group* g = nullptr;
            void finish() { if (pool) { pool->wait(g); pool = nullptr; } }
            ~DrainGuard() { finish(); }
        } drain_guard;
        if (s.pending_dst && s.pending_bytes >= (4u << 20) && !in_pinned) {
            if (!copy_pool) copy_pool = make_copy_pool();
            copy_pool->start(s.pending_dst, s.h_out, s.pending_bytes, &drain);
            drain_guard.pool = copy_pool; drain_guard.g = &drain;
            s.pending_dst = nullptr; s.pending_bytes = 0;
        } else {
            flush_pending(s);
        }
        const uint64_t nf = std::min<uint64_t>(fpc, p.n_frames - f0);
        const uint64_t s_begin = p.start_sample + f0 * p.hop;
        uint64_t s_end = s_begin + (nf - 1) * p.hop + p.nfft;
        if (s_end > n_samples) s_end = n_samples;             // frames past EOF become fill rows
        const uint64_t ns = s_end > s_begin ? s_end - s_begin : 0;
        if (ns && !no_data) {
            const void* src = (const char*)iq + s_begin * bps;
            if (hs.fd >= 0) {                                  // parallel pread straight into the pinned ring
                if (!host_read(s.h_in, hs.fd, hs.file_off + s_begin * bps, ns * bps)) {
                    rc = set_error(SA_ERR_OUT_OF_RANGE, "short read at byte %llu of the data file",
                                   (unsigned long long)(hs.file_off + s_begin * bps));
                    break;
                }
                src = s.h_in;
            } else if (!in_pinned) { host_copy(s.h_in, src, ns * bps); src = s.h_in; }
            e = cudaMemcpyAsync(s.d_in, src, ns * bps, cudaMemcpyHostToDevice, s.stream);
            if (e != cudaSuccess) { rc = cuda_fail(e, "H2D"); break; }
        }
        drain_guard.finish();                                // h_out is free before this chunk's D2H is queued
        sa_spectrogram_params q = p;
        q.start_sample = 0;
        q.n_frames = nf;
        rc = launch_spectrogram(s.d_in, ns, q, prec, s.d_out, s.stream, 5 + (int)(c % kSlots));
        if (rc) break;
        void* dst = (char*)out + f0 * row_bytes;
        if (!out_pinned) { s.pending_dst = dst; s.pending_bytes = nf * row_bytes; dst = s.h_out; }
        e = cudaMemcpyAsync(dst, s.d_out, nf * row_bytes, cudaMemcpyDeviceToHost, s.stream);
        if (e != cudaSuccess) { rc = cuda_fail(e, "D2H"); break; }
    }
    for (int i = 0; i < kSlots; i++)
        if (slots[i].stream) {
            cudaError_t e = cudaStreamSynchronize(slots[i].stream);
            if (e != cudaSuccess && rc == SA_OK) rc = cuda_fail(e, "pipeline drain");
            if (rc == SA_OK) flush_pending(slots[i]);
            slots[i].pending_dst = nullptr;
        }
    return rc;
}

Engine::~Engine() {
    cudaSetDevice(device);
    for (auto& kv : twiddles) cudaFree(kv.second);
    for (auto& kv : windows) cudaFree(kv.second);
    for (auto& kv : misc_tables) cudaFree(kv.second);
    for (int i = 0; i < kSlots; i++) {
        if (slots[i].d_in) cudaFree(slots[i].d_in);
        if (slots[i].d_out) cudaFree(slots[i].d_out);
        if (slots[i].stream) cudaStreamDestroy(slots[i].stream);
        if (slots[i].h_in) cudaFreeHost(slots[i].h_in);
        if (slots[i].h_out) cudaFreeHost(slots[i].h_out);
    }
    for (int i = 0; i < 4; i++) {
        if (large_aux[i]) cudaStreamDestroy(large_aux[i]);
        for (int j = 0; j < 2; j++) if (large_ev[i][j]) cudaEventDestroy(large_ev[i][j]);
    }
    if (h_plan) cudaFreeHost(h_plan);
    if (plan_ev) cudaEventDestroy(plan_ev);
    if (dc_aux) cudaStreamDestroy(dc_aux);
    for (int j = 0; j < 2; j++) if (dc_ev[j]) cudaEventDestroy(dc_ev[j]);
    for (int j = 0; j < 4; j++) if (dc_pipe_ev[j]) cudaEventDestroy(dc_pipe_ev[j]);
    delete copy_pool;
    for (auto& r : registered) cudaHostUnregister(const_cast<void*>(r));
    for (int i = 0; i < kScratch; i++) if (scratch[i]) cudaFree(scratch[i]);
}

int Engine::ensure_scratch(int which, size_t bytes) {
    if (scratch_cap[which] >= bytes) return SA_OK;
    if (scratch[which]) { cudaDeviceSynchronize(); cudaFree(scratch[which]); }
    scratch[which] = nullptr; scratch_cap[which] = 0;
    cudaError_t e = cudaMalloc(&scratch[which], bytes);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMalloc(scratch)");
    scratch_cap[which] = bytes;
    return SA_OK;
}

}  // namespace sa

using namespace sa;



extern "C" {

const char* sa_last_error(void) { return g_err; }
const char* sa_version(void) { return "spectral_analyzer_b200 0.1.0 (sm_100a)"; }

int32_t sa_bytes_per_iq(int32_t dtype) {     // S/sigmf/Global.java:67-79
    switch (dtype) {
        case SA_CF32: return 8;
        case SA_CI16: return 4;
        case SA_CU8:  return 2;
        case SA_CI8:  return 2;
        case SA_CF64: return 16;
        default:      return 0;
    }
}

int32_t sa_parse_datatype(const char* s, int32_t* dtype, int32_t* big_endian) {
    if (!s || !dtype || !big_endian) return set_error(SA_ERR_INVALID_ARG, "NULL argument");
    // String.startsWith tests of SpectralService.java:35-38 / ExtractDownConvertService.java:79-94
    int d = -1;
    if (!strncmp(s, "ci16", 4)) d = SA_CI16;
    else if (!strncmp(s, "cf32", 4)) d = SA_CF32;
    else if (!strncmp(s, "cu8", 3)) d = SA_CU8;
    else if (!strncmp(s, "ci8", 3)) d = SA_CI8;
    else if (!strncmp(s, "cf64", 4)) d = SA_CF64;
    if (d < 0) return set_error(SA_ERR_UNSUPPORTED, "datatype '%s' has no decode branch", s);
    const size_t n = strlen(s);
    *big_endian = (n >= 3 && !strcmp(s + n - 3, "_le")) ? 0 : 1;     // SigMfHelper.java:87-91
    *dtype = d;
    return SA_OK;
}

void sa_spectrogram_params_init(sa_spectrogram_params* p) {
    if (!p) return;
    memset(p, 0, sizeof(*p));
    p->struct_size = sizeof(*p);
    p->dtype = SA_CF32;
    p->window = SA_WIN_RECT;
    p->nfft = 1024;                 // main-scene.fxml:129-132 default 2^10
    p->db_mode = SA_DB_MAG_1E10;
    p->out_kind = SA_OUT_F32_DB;
    p->precision = SA_PREC_AUTO;
    p->hop = 1024;
    p->eof_fill_db = -150.0;        // MainController.java:996-997
    p->colormap = SA_CMAP_GRAYSCALE;
    p->sample_rate = 1.0;
    p->min_db = -160.0;             // main-scene.fxml:143
    p->max_db = -30.0;              // main-scene.fxml:150
}

int32_t sa_engine_create(int32_t device, sa_engine** out) {
    if (!out) return set_error(SA_ERR_INVALID_ARG, "out_engine is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return set_error(SA_ERR_NO_DEVICE, "no CUDA device (%s); this engine has no CPU fallback",
                         e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= count) return set_error(SA_ERR_INVALID_ARG, "device %d out of range (count %d)", device, count);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceProperties");
    if (prop.major != 10)
        return set_error(SA_ERR_NO_DEVICE, "device %d is sm_%d%d; this library carries sm_100a code only", device, prop.major, prop.minor);
    sa_engine* eng = new sa_engine();
    eng->device = device;
    eng->num_sms = prop.multiProcessorCount;
    const char* cm = getenv("SA_CHUNK_MB");
    if (cm && atoi(cm) > 0) eng->chunk_bytes = (uint64_t)atoi(cm) << 20;
    *out = eng;
    return SA_OK;
}

void sa_engine_destroy(sa_engine* engine) {
    if (!engine) return;
    { std::lock_guard<std::mutex> lock_(engine->mu); cudaSetDevice(engine->device); cudaDeviceSynchronize(); }
    delete engine;
}

uint64_t sa_kernel_launches(const sa_engine* engine) { return engine ? engine->launches : 0; }

int32_t sa_register_host(sa_engine* engine, const void* ptr, uint64_t bytes, int32_t read_only) {
    ENGINE_ENTER(engine);
    if (!ptr || !bytes) return set_error(SA_ERR_INVALID_ARG, "empty range");
    unsigned flags = cudaHostRegisterPortable;
    if (read_only) flags |= cudaHostRegisterReadOnly;
    cudaError_t e = cudaHostRegister(const_cast<void*>(ptr), bytes, flags);
    if (e != cudaSuccess && read_only) {      // some platforms refuse the read-only flag
        cudaGetLastError();
        e = cudaHostRegister(const_cast<void*>(ptr), bytes, cudaHostRegisterPortable);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return set_error(SA_ERR_CUDA, "cudaHostRegister: %s (file-backed mappings cannot be page-locked; unregistered "
                         "buffers are staged through pinned memory by the engine)", cudaGetErrorString(e));
    }
    engine->registered.push_back(ptr);
    return SA_OK;
}

int32_t sa_unregister_host(sa_engine* engine, const void* ptr) {
    ENGINE_ENTER(engine);
    auto it = std::find(engine->registered.begin(), engine->registered.end(), ptr);
    if (it == engine->registered.end()) return set_error(SA_ERR_INVALID_ARG, "range was not registered");
    engine->registered.erase(it);
    cudaError_t e = cudaHostUnregister(const_cast<void*>(ptr));
    if (e != cudaSuccess) return cuda_fail(e, "cudaHostUnregister");
    return SA_OK;
}

int32_t sa_spectrogram_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes,
                              const sa_spectrogram_params* params, void* d_out, uint64_t out_bytes,
                              void* cuda_stream) {
    ENGINE_ENTER(engine);
    int prec = 0;
    int rc = check_spec_params(params, &prec);
    if (rc) return rc;
    if (!d_out || (!d_iq && iq_bytes)) return set_error(SA_ERR_INVALID_ARG, "NULL buffer");
    const uint64_t bps = spec_bytes_per_iq(*params);
    if ((uintptr_t)d_iq % bps) return set_error(SA_ERR_INVALID_ARG, "d_iq must be aligned to %llu bytes", (unsigned long long)bps);
    const uint64_t need = params->n_frames * (uint64_t)params->nfft * out_elem_bytes(params->out_kind);
    if (out_bytes < need) return set_error(SA_ERR_SMALL_OUTPUT, "out_bytes %llu < %llu", (unsigned long long)out_bytes, (unsigned long long)need);
    return engine->launch_spectrogram(d_iq, iq_bytes / bps, *params, prec, d_out, (cudaStream_t)cuda_stream);
}

int32_t sa_spectrogram(sa_engine* engine, const void* iq, uint64_t iq_bytes, const sa_spectrogram_params* params,
                       void* out, uint64_t out_bytes) {
    ENGINE_ENTER(engine);
    int prec = 0;
    int rc = check_spec_params(params, &prec);
    if (rc) return rc;
    if (!out || (!iq && iq_bytes)) return set_error(SA_ERR_INVALID_ARG, "NULL buffer");
    const uint64_t need = params->n_frames * (uint64_t)params->nfft * out_elem_bytes(params->out_kind);
    if (out_bytes < need) return set_error(SA_ERR_SMALL_OUTPUT, "out_bytes %llu < %llu", (unsigned long long)out_bytes, (unsigned long long)need);
    if (params->n_frames == 0) return SA_OK;
    HostSource hs;
    hs.ptr = iq;
    return engine->spectrogram_host(hs, iq_bytes, *params, prec, out);
}

// File-based ingest (SigMfHelper.load, S/sigmf/SigMfHelper.java:59-84: the data file, core:header_bytes skipped):
// the samples go from the page cache / the device straight into the pinned ring by parallel pread, without the
// page-fault + memcpy hop of an mmapped buffer, and without the reference's 2 GiB mapping limit (:78-82).
int32_t sa_spectrogram_file(sa_engine* engine, const char* path, uint64_t data_offset, uint64_t data_bytes,
                            const sa_spectrogram_params* params, void* out, uint64_t out_bytes) {
    ENGINE_ENTER(engine);
    int prec = 0;
    int rc = check_spec_params(params, &prec);
    if (rc) return rc;
    if (!path || !out) return set_error(SA_ERR_INVALID_ARG, "NULL path / buffer");
    const uint64_t need = params->n_frames * (uint64_t)params->nfft * out_elem_bytes(params->out_kind);
    if (out_bytes < need) return set_error(SA_ERR_SMALL_OUTPUT, "out_bytes %llu < %llu", (unsigned long long)out_bytes, (unsigned long long)need);
    const int fd = open(path, O_RDONLY | O_CLOEXEC);
    if (fd < 0) return set_error(SA_ERR_INVALID_ARG, "cannot open '%s': %s", path, strerror(errno));
    struct stat st;
    if (fstat(fd, &st) != 0) { close(fd); return set_error(SA_ERR_INVALID_ARG, "fstat '%s': %s", path, strerror(errno)); }
    const uint64_t size = (uint64_t)st.st_size;
    if (data_offset > size) { close(fd); return set_error(SA_ERR_OUT_OF_RANGE, "data_offset %llu beyond the %llu-byte file", (unsigned long long)data_offset, (unsigned long long)size); }
    uint64_t avail = size - data_offset;
    if (data_bytes && data_bytes < avail) avail = data_bytes;          // one capture of a multi-capture recording
    if (params->n_frames == 0) { close(fd); return SA_OK; }
    HostSource hs;
    hs.fd = fd;
    hs.file_off = data_offset;
    rc = engine->spectrogram_host(hs, avail, *params, prec, out);
    close(fd);
    return rc;
}

const char* sa_last_kernel_name(sa_engine* engine) {
    static thread_local std::string name;
    if (!engine) return "";
    std::lock_guard<std::mutex> lock_(engine->mu);
    name = engine->last_kernel;
    return name.c_str();
}

int32_t sa_compute_magnitudes(sa_engine* engine, const void* buffer, uint64_t capacity_bytes, uint64_t start_byte,
                              uint32_t nfft, int32_t dtype, int32_t big_endian, double* out) {
    ENGINE_ENTER(engine);
    sa_spectrogram_params p;
    sa_spectrogram_params_init(&p);
    p.dtype = dtype; p.big_endian = big_endian; p.nfft = nfft; p.hop = nfft; p.n_frames = 1;
    p.out_kind = SA_OUT_F64_DB;
    p.strict_reference = engine->profile.strict_reference;      // the engine's profile: zeros for cf64 / unknown datatypes
    int prec = 0;
    int rc = check_spec_params(&p, &prec);
    if (rc) return rc;
    if (!buffer || !out) return set_error(SA_ERR_INVALID_ARG, "NULL buffer");
    const uint64_t bps = spec_bytes_per_iq(p);
    // buffer.getShort/getFloat past the limit throws IndexOutOfBoundsException in Java (nothing is read for the
    // datatypes that decode to zeros)
    if (!strict_zero(p) && (start_byte > capacity_bytes || (uint64_t)nfft * bps > capacity_bytes - start_byte))
        return set_error(SA_ERR_OUT_OF_RANGE, "frame [%llu, +%llu) exceeds capacity %llu", (unsigned long long)start_byte,
                         (unsigned long long)(nfft * bps), (unsigned long long)capacity_bytes);
    HostSource hs;
    hs.ptr = (const char*)buffer + (strict_zero(p) ? 0 : start_byte);
    return engine->spectrogram_host(hs, (uint64_t)nfft * bps, p, prec, out);
}

}  // extern "C"
