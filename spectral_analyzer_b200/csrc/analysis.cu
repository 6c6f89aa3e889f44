// analysis.cu -- annotation-analysis path behind the C-ABI: NCO downconvert + FIR decimate and
// Welch PSD (kernels in analysis_kernels.cuh).  Replaces ExtractDownConvertService.java:54-117,
// the batch loop AnnotationController.java:321-360 and the calculatePsdWelch call at
// AnalysisDialogController.java:308-312.  Everything JDSP decides inside those calls (not vendored,
// build.gradle:142) is a field of the engine's analysis profile (sa_analysis_config).
#include "engine_internal.h"
#include "analysis_kernels.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <tuple>

using namespace sa;


namespace {

const double kPi = 3.14159265358979323846264338327950288;

// Hamming-windowed sinc, ntaps = 8*down+1, cutoff 0.5/down cycles/sample, unity DC gain
void lowpass_taps(int down, std::vector<double>& h) {
    const int nt = 8 * down + 1, mid = 4 * down;
    const double fc = 0.5 / down;
    h.resize(nt);
    double sum = 0.0;
    for (int k = 0; k < nt; k++) {
        const double x = (double)(k - mid);
        const double s = (k == mid) ? 2.0 * fc : std::sin(2.0 * kPi * fc * x) / (kPi * x);
        const double w = 0.54 - 0.46 * std::cos(2.0 * kPi * (double)k / (double)(nt - 1));
        h[k] = s * w;
        sum += h[k];
    }
    for (int k = 0; k < nt; k++) h[k] /= sum;
}

struct WelchKernel { const void* fn; const void* fin; int prec, n, cta, fpc; size_t smem; int p, np, radix[4]; int mid; int slots; };   // slots: partial spectra a CTA writes

template <typename T, int N> WelchKernel make_welch(int prec) {
    using G = Geo<T, N>;
    using PL = Plan<T, N>;
    WelchKernel k;
    k.fn = (const void*)&welch_accum_kernel<T, N>;
    k.fin = (const void*)&welch_finalize_kernel<T>;
    k.prec = prec;
    k.n = N; k.cta = G::CTA; k.fpc = G::FPC; k.smem = G::SMEM_BYTES + G::TW_BYTES; k.p = G::P; k.np = PL::NP;
    for (int i = 0; i < 4; i++) k.radix[i] = PL::radix(i);
    k.mid = 0;
    k.slots = k.fpc;
    return k;
}
// FP32 2048 .. 16384: the small-radix-first plan (welch_accum_mid_kernel)
template <int N, int CTA_ = MidGeo<N>::CTA> WelchKernel make_welch_mid() {
    using G = MidGeo<N>;
    WelchKernel k;
    k.fn = (const void*)&welch_accum_mid_kernel<N, CTA_>;
    k.fin = (const void*)&welch_finalize_kernel<float>;
    k.prec = 1;
    k.n = N; k.cta = CTA_; k.fpc = CTA_ / G::TPF;
    k.smem = (size_t)k.fpc * G::SM_ELEMS * sizeof(float2) + G::T1_BYTES + G::WIN_BYTES; k.p = 32; k.np = 3;
    k.radix[0] = G::R0; k.radix[1] = 32; k.radix[2] = 32; k.radix[3] = 1;
    k.mid = 1;
    k.slots = 1;                 // the CTA adds up its segment slots itself
    return k;
}

const WelchKernel* find_welch(int prec, int n) {
    static const bool no_mid = getenv("SA_WELCH_MID") && atoi(getenv("SA_WELCH_MID")) == 0;     // A/B: the general plan
    static const WelchKernel mid_tab[] = { make_welch_mid<2048>(), make_welch_mid<4096>(), make_welch_mid<8192>(), make_welch_mid<16384>() };
    // SA_WELCH_CTA=256: one segment per CTA for 8192 points (256 threads, 32 K registers), small enough to share an SM with
    // the row-per-thread downconverter's CTAs when the batches are pipelined (run_batch_device); measured no faster
    static const bool small_cta = getenv("SA_WELCH_CTA") && atoi(getenv("SA_WELCH_CTA")) == 256;
    static const WelchKernel mid_8192_small = make_welch_mid<8192, 256>();
    if (prec == 1 && !no_mid && n == 8192 && small_cta) return &mid_8192_small;
    if (prec == 1 && !no_mid)
        for (const auto& k : mid_tab) if (k.n == n) return &k;
    static const WelchKernel tab[] = {
        make_welch<float, 64>(1), make_welch<float, 128>(1), make_welch<float, 256>(1), make_welch<float, 512>(1),
        make_welch<float, 1024>(1), make_welch<float, 2048>(1), make_welch<float, 4096>(1), make_welch<float, 8192>(1),
        make_welch<float, 16384>(1),
        make_welch<double, 64>(2), make_welch<double, 128>(2), make_welch<double, 256>(2), make_welch<double, 512>(2),
        make_welch<double, 1024>(2), make_welch<double, 2048>(2), make_welch<double, 4096>(2), make_welch<double, 8192>(2) };
    for (const auto& k : tab) if (k.prec == prec && k.n == n) return &k;
    return nullptr;
}

// which: 0 staged kernel with taps from global memory, 1 staged kernel with taps in the parameter bank,
// 2 warp-per-output kernel, 3 pipelined staged kernel (taps in the parameter bank)
template <int DK> const void* dc_kernel_of(int which) {
    if (which == 2) return (const void*)&downconvert_wide_kernel<DK>;
    if (which == 1) return (const void*)&downconvert_kernel<DK, true, false>;
    if (which == 3) {
        if constexpr (sizeof(typename DcRaw<DK>::raw_t) <= 8) return (const void*)&downconvert_kernel<DK, true, true>;
        else return nullptr;
    }
    return (const void*)&downconvert_kernel<DK, false, false>;
}
const void* dc_kernel(int dk, int which) {
    switch (dk) {
        case DK_CF32: return dc_kernel_of<DK_CF32>(which);
        case DK_CI16: return dc_kernel_of<DK_CI16>(which);
        case DK_C8:   return dc_kernel_of<DK_C8>(which);
        case DK_CF64_S8: return dc_kernel_of<DK_CF64_S8>(which);
        default:      return dc_kernel_of<DK_CF64>(which);
    }
}

// row-per-thread kernel (cf32, little-endian, power-of-two decimation): nullptr when there is none for this factor.
// mode 0: taps and NCO phasors as shared-memory tables, FFMA2; mode 1: taps as constant-bank immediates, NCO recurrence
struct DcRowsShape { int mode, nt, nbuf, swz; };
// Shape of the row kernel, measured on B200 (C3 = 500 x 2^20 samples at D 16 incl. Welch; tools/dc_matrix.py for 8 / 32):
//   rows per tile x raw buffers     C3          D 8        D 16       D 32
//   256 x 1                          1.413 ms    0.827      0.621      0.479
//   256 x 2                          1.407       0.805      0.617      0.580
//   128 x 1                          1.464       0.793      0.634      0.457
//   128 x 2                          1.325       0.784      0.581      0.507
// (small tiles double-buffered: every CTA always has a tile in flight and the load / tap-loop phases of the resident
// CTAs no longer line up; at D 32 two buffers cost too many CTAs).  SA_DC_ROWS_NT / SA_DC_ROWS_NBUF / SA_DC_ROWS_MODE override.
static DcRowsShape dc_rows_shape(int dk, int down) {
    static const char* me = getenv("SA_DC_ROWS_MODE");
    static const char* ne = getenv("SA_DC_ROWS_NT");
    static const char* be = getenv("SA_DC_ROWS_NBUF");
    static const char* se = getenv("SA_DC_ROWS_SWZ");
    DcRowsShape sh = { me ? atoi(me) : 1, ne ? atoi(ne) : 128, be ? atoi(be) : (down >= 32 ? 1 : 2), se ? atoi(se) : 1 };
    if (sh.nt != 256) sh.nt = 128;
    if (sh.nbuf != 1) sh.nbuf = 2;
    if (sh.mode == 0) { sh.nt = 256; sh.nbuf = 1; sh.swz = 0; }
    if (dk != DK_CF32) { sh.mode = 1; sh.nt = 128; }       // the integer types exist in the 128-row shapes only
    {
        const int cpr = down / (dk == DK_CF32 ? 2 : (dk == DK_CI16 ? 4 : 8));
        if (cpr & (cpr - 1)) { sh.mode = 1; sh.nt = 128; sh.swz = 0; }     // 3, 5, 6, 7 ... chunks per row: 128-row shapes, no swizzle
    }
    if (sh.nt == 256) sh.swz = 0;                          // swizzled rows exist in the 128-row shapes (256 x 2 swizzled: C3 1.268 ms against 1.231)        // the table variant exists in the first shape only (ablation record)
    return sh;
}
template <int DK, int D, int NT, int NBUF, bool SWZ = false> const void* dc_rows_fn(size_t* smem) {
    *smem = DcRowsGeo<D, NT, NBUF, DcRowsSpc<DK>::value, SWZ>::SMEM;
    return (const void*)&downconvert_rows_kernel<DK, D, 1, NT, NBUF, SWZ>;
}
// cf32: every shape (the A/B record of dc_rows_shape) and the table variant; the integer types: the default shapes only
template <int DK, int D> const void* dc_rows_kernel_of(const DcRowsShape& sh, size_t* smem) {
    if constexpr (D % DcRowsSpc<DK>::value != 0) { *smem = 0; return nullptr; }
    else if constexpr (DK == DK_CF32) {
        if (sh.mode == 0) { *smem = DcRowsGeo<D, 256, 1>::SMEM; return (const void*)&downconvert_rows_kernel<DK_CF32, D, 0, 256, 1, false>; }
        if (sh.nt == 256 && sh.nbuf == 1) return dc_rows_fn<DK, D, 256, 1>(smem);
        if (sh.nt == 256 && sh.nbuf == 2) return dc_rows_fn<DK, D, 256, 2>(smem);
        if (sh.nt == 128 && sh.nbuf == 1) return sh.swz ? dc_rows_fn<DK, D, 128, 1, true>(smem) : dc_rows_fn<DK, D, 128, 1>(smem);
        return sh.swz ? dc_rows_fn<DK, D, 128, 2, true>(smem) : dc_rows_fn<DK, D, 128, 2>(smem);
    } else {
        if (sh.nbuf == 1) return sh.swz ? dc_rows_fn<DK, D, 128, 1, true>(smem) : dc_rows_fn<DK, D, 128, 1>(smem);
        return sh.swz ? dc_rows_fn<DK, D, 128, 2, true>(smem) : dc_rows_fn<DK, D, 128, 2>(smem);
    }
}
// decimations whose rows are a power-of-two number of chunks come in every shape; the other even ones (cf32: 6, 10, 12 ... 30;
// ci16: 12, 20, 24, 28; cu8 / ci8: 24) in the 128-row shapes with packed (odd chunk count) or padded rows
template <int DK, int D> const void* dc_rows_kernel_np2(const DcRowsShape& sh, size_t* smem) {
    if constexpr (D % DcRowsSpc<DK>::value != 0) { *smem = 0; return nullptr; }
    else return sh.nbuf == 1 ? dc_rows_fn<DK, D, 128, 1>(smem) : dc_rows_fn<DK, D, 128, 2>(smem);
}
template <int DK> const void* dc_rows_kernel_dk(int down, const DcRowsShape& sh, size_t* smem) {
    switch (down) {
        case 4:  return dc_rows_kernel_of<DK, 4>(sh, smem);
        case 8:  return dc_rows_kernel_of<DK, 8>(sh, smem);
        case 16: return dc_rows_kernel_of<DK, 16>(sh, smem);
        case 32: return dc_rows_kernel_of<DK, 32>(sh, smem);
        case 6:  return dc_rows_kernel_np2<DK, 6>(sh, smem);
        case 10: return dc_rows_kernel_np2<DK, 10>(sh, smem);
        case 12: return dc_rows_kernel_np2<DK, 12>(sh, smem);
        case 14: return dc_rows_kernel_np2<DK, 14>(sh, smem);
        case 18: return dc_rows_kernel_np2<DK, 18>(sh, smem);
        case 20: return dc_rows_kernel_np2<DK, 20>(sh, smem);
        case 22: return dc_rows_kernel_np2<DK, 22>(sh, smem);
        case 24: return dc_rows_kernel_np2<DK, 24>(sh, smem);
        case 26: return dc_rows_kernel_np2<DK, 26>(sh, smem);
        case 28: return dc_rows_kernel_np2<DK, 28>(sh, smem);
        case 30: return dc_rows_kernel_np2<DK, 30>(sh, smem);
        default: *smem = 0; return nullptr;
    }
}
const void* dc_rows_kernel(int dk, int down, const DcRowsShape& sh, size_t* smem) {
    switch (dk) {
        case DK_CF32: return dc_rows_kernel_dk<DK_CF32>(down, sh, smem);
        case DK_CI16: return dc_rows_kernel_dk<DK_CI16>(down, sh, smem);
        case DK_C8:   return dc_rows_kernel_dk<DK_C8>(down, sh, smem);
        default: *smem = 0; return nullptr;
    }
}
const void* dc_rows_fast_kernel(int dk) {
    switch (dk) {
        case DK_CF32: return (const void*)&downconvert_rows_fast_kernel<DK_CF32>;
        case DK_CI16: return (const void*)&downconvert_rows_fast_kernel<DK_CI16>;
        case DK_C8:   return (const void*)&downconvert_rows_fast_kernel<DK_C8>;
        default: return nullptr;
    }
}
static bool dc_rows_aligned(long long first, long long spc) { const long long r = first & (spc - 1); return r == 0 || r == spc - 1; }
// kernel-parameter tap block of the row kernel (the layout of DcRowsTaps<D>): g[sg][i][p] = h[(p+1)D - i - sg], h[0], h[8D]
static void dc_rows_taps(const float* h, int D, std::vector<float>& out) {
    out.assign((size_t)2 * D * 8 + 4, 0.f);
    for (int sg = 0; sg < 2; sg++)
        for (int i = 0; i < D; i++)
            for (int p = 0; p < 8; p++) out[((size_t)sg * D + i) * 8 + p] = h[(p + 1) * D - i - sg];
    out[(size_t)2 * D * 8] = h[0];
    out[(size_t)2 * D * 8 + 1] = h[8 * D];
}

size_t dc_smem_bytes(int down, int nb, int fast, bool pipe) {
    const int nblk = nb + (fast ? 0 : 7);
    const size_t n_stage = fast ? (size_t)nb * down : (size_t)nblk * down + 1;
    const size_t stage_phys = n_stage + n_stage / down + 2;
    return ((stage_phys + 1) & ~(size_t)1) * sizeof(float2) + (fast ? 0 : (size_t)nblk * 8 * sizeof(float2)) +
           (pipe ? (size_t)dc_tap_smem_bytes(down) : 0);
}

int validate_anns(const sa_annotation* anns, uint32_t n_ann, uint64_t n_samples, uint64_t extra) {
    if (!anns && n_ann) return set_error(SA_ERR_INVALID_ARG, "annotations is NULL");
    for (uint32_t i = 0; i < n_ann; i++) {
        if (anns[i].down < 1) return set_error(SA_ERR_INVALID_ARG, "annotation %u: down %d < 1", i, anns[i].down);
        if (!std::isfinite(anns[i].freq_off)) return set_error(SA_ERR_INVALID_ARG, "annotation %u: freq_off not finite", i);
        const uint64_t need = anns[i].count ? anns[i].count + extra : 0;
        if (anns[i].start_sample > n_samples || need > n_samples - anns[i].start_sample)
            return set_error(SA_ERR_OUT_OF_RANGE, "annotation %u: [%llu, +%llu) exceeds %llu samples", i,
                             (unsigned long long)anns[i].start_sample, (unsigned long long)anns[i].count,
                             (unsigned long long)n_samples);
    }
    return SA_OK;
}

}  // namespace

namespace sa {

// taps in effect for decimation factor `down` (profile taps, or the built-in design)
static void profile_taps(const AnalysisProfile& pf, int down, std::vector<double>& h) {
    if (!pf.taps.empty()) h = pf.taps; else lowpass_taps(down, h);
}

// number of outputs (DESIGN.md K5)
uint64_t dc_out_len(const AnalysisProfile& pf, uint64_t count, int down, int fast) {
    const uint64_t L = pf.taps.empty() ? 8ull * (uint64_t)down + 1 : pf.taps.size();
    if (!fast && pf.delay_mode == SA_DELAY_VALID) return count >= L ? (count - L) / (uint64_t)down + 1 : 0;
    return pf.length_mode == SA_LEN_CEIL ? (count + (uint64_t)down - 1) / (uint64_t)down : count / (uint64_t)down;
}

struct WelchJob { const double* re; const double* im; const float2* f32; long long n; double fs; double* d_out; };

// One Welch launch: all signals share the transform length.  Prepared on the host first (so that every plan of a
// call can be uploaded in ONE copy before the first kernel is launched: a pageable H2D copy in the middle of the
// launch sequence synchronises the stream and serialises everything behind it), launched later.
struct WelchLaunch {
    std::vector<WelchSig> sigs;
    std::vector<double*> d_out;
    const WelchKernel* wk = nullptr;
    uint32_t nfft = 0;
    uint64_t hop = 0;
    int window = 0, prec = SA_PREC_F32, nsplit = 1;
    size_t direct_smem = 0;
};

static int welch_prepare(Engine* eng, const std::vector<WelchJob>& jobs, uint32_t nfft, uint64_t hop, int window, WelchLaunch& wl) {
    const AnalysisProfile& pf = eng->profile;
    wl.prec = pf.psd_precision == SA_PREC_F64 ? SA_PREC_F64 : SA_PREC_F32;
    const size_t elem = wl.prec == SA_PREC_F64 ? 8 : 4;
    const bool pow2 = nfft >= 64 && (nfft & (nfft - 1)) == 0;
    wl.wk = pow2 ? find_welch(wl.prec, (int)nfft) : nullptr;
    wl.direct_smem = ((size_t)nfft + kDirectTile) * 2 * elem;
    if (!wl.wk && wl.direct_smem > 200 * 1024)
        return set_error(SA_ERR_UNSUPPORTED, "psd nfft %u: %s transforms go up to %d points (powers of two) or %d points (any length)",
                         nfft, wl.prec == SA_PREC_F64 ? "FP64" : "FP32", wl.prec == SA_PREC_F64 ? 8192 : 16384,
                         (int)(200 * 1024 / (2 * elem)) - kDirectTile);
    const uint32_t n_sig = (uint32_t)jobs.size();
    if (n_sig > 65535) return set_error(SA_ERR_UNSUPPORTED, "more than 65535 signals in one PSD launch");
    wl.nfft = nfft; wl.hop = hop; wl.window = window;
    std::vector<double> w;
    host_window(window, (int)nfft, w);
    double sw = 0.0, sw2 = 0.0;
    for (double v : w) { sw += v; sw2 += v * v; }
    wl.sigs.resize(n_sig);
    wl.d_out.resize(n_sig);
    long long max_seg = 0;
    for (uint32_t i = 0; i < n_sig; i++) {
        WelchSig& s = wl.sigs[i];
        s.re = jobs[i].re; s.im = jobs[i].im; s.f32 = jobs[i].f32; s.n = jobs[i].n;
        s.nseg = s.n >= (long long)nfft ? 1 + (s.n - nfft) / (long long)hop : 0;
        const double den = pf.psd_scaling == SA_PSD_SPECTRUM ? sw * sw : jobs[i].fs * sw2;
        s.scale = s.nseg > 0 ? 1.0 / ((double)s.nseg * den) : 0.0;
        max_seg = std::max(max_seg, s.nseg);
        wl.d_out[i] = jobs[i].d_out;
    }
    // CTAs per signal: about four segments per frame slot, whatever else is in the launch (the summation order of a
    // signal then depends only on its own launch's longest signal, not on how many signals share the launch)
    wl.nsplit = 1;
    static const char* steps_env = getenv("SA_WELCH_STEPS");                 // segments per slot (A/B switch)
    const long long steps = steps_env && atoi(steps_env) > 0 ? atoi(steps_env) : 8;    // C3: 4 -> 8: 1.224 -> 1.172 ms (fewer partial spectra and finalize reads)
    if (wl.wk) wl.nsplit = (int)std::max<long long>(1, std::min<long long>(64, (max_seg + steps * wl.wk->fpc - 1) / (steps * wl.wk->fpc)));
    return SA_OK;
}

// d_sigs: the launch's WelchSig array on the device (already uploaded, or NULL: uploaded here from pageable memory).
// `wsi` selects one of two workspaces (batches alternate between two streams).
static int welch_launch(Engine* eng, const WelchLaunch& wl, const WelchSig* d_sigs, cudaStream_t stream, int wsi) {
    const AnalysisProfile& pf = eng->profile;
    const uint32_t n_sig = (uint32_t)wl.sigs.size(), nfft = wl.nfft;
    if (n_sig == 0) return SA_OK;
    const size_t elem = wl.prec == SA_PREC_F64 ? 8 : 4;
    const WelchKernel* wk = wl.wk;
    const size_t sig_bytes = d_sigs ? 0 : (((size_t)n_sig * sizeof(WelchSig) + 255) & ~(size_t)255);
    // consecutive destination rows: the kernels write them in place; otherwise packed rows + one copy per run
    bool contiguous = wl.d_out[0] != nullptr;
    for (uint32_t i = 1; i < n_sig && contiguous; i++) contiguous = wl.d_out[i] == wl.d_out[i - 1] + nfft;
    const size_t out_bytes = contiguous ? 0 : (((size_t)n_sig * nfft * sizeof(double) + 255) & ~(size_t)255);
    const size_t part_bytes = wk ? (size_t)n_sig * wl.nsplit * wk->slots * nfft * elem : 0;
    const int slot = wsi ? 9 : 1;
    int rc = eng->ensure_scratch(slot, std::max<size_t>(sig_bytes + out_bytes + part_bytes, 256) + 256);      // + the task counter
    if (rc) return rc;
    char* base = (char*)eng->scratch[slot];
    double* d_rows = (double*)(base + sig_bytes);
    cudaError_t e = cudaSuccess;
    if (!d_sigs) {
        // pageable source: the driver has staged the bytes when the call returns
        e = cudaMemcpyAsync(base, wl.sigs.data(), wl.sigs.size() * sizeof(WelchSig), cudaMemcpyHostToDevice, stream);
        if (e != cudaSuccess) return cuda_fail(e, "upload Welch plan");
        d_sigs = (const WelchSig*)base;
    }
    WelchArgs wa;
    memset(&wa, 0, sizeof(wa));
    wa.sigs = d_sigs;
    wa.hop = (long long)wl.hop;
    wa.detrend = pf.psd_detrend == SA_DETREND_CONSTANT ? 1 : 0;
    wa.window_id = wl.window;
    wa.out_db = contiguous ? wl.d_out[0] : d_rows;
    if (wk) {
        SpecKernelInfo ki;
        memset(&ki, 0, sizeof(ki));
        ki.prec = wl.prec; ki.n = wk->n; ki.p = wk->p; ki.np = wk->np;
        for (int i = 0; i < 4; i++) ki.radix[i] = wk->radix[i];
        if (wk->mid) {
            rc = eng->mid_t1_table(wk->n, &wa.twiddle);
            if (rc) return rc;
            rc = eng->root_table(wk->n, wl.prec, &wa.aux);
        } else {
            rc = eng->twiddle_table(ki, &wa.twiddle);
        }
        if (rc) return rc;
        rc = eng->window_table(wl.window, (int)nfft, wl.prec, &wa.window);
        if (rc) return rc;
        wa.partial = base + sig_bytes + out_bytes;
        wa.nsplit = wl.nsplit;
        int bps = 0;
        rc = eng->kernel_grid(wk->fn, wk->cta, wk->smem, &bps);
        if (rc) return rc;
        void* wargs[] = { &wa };
        dim3 grid(wl.nsplit, n_sig);
        if (wk->mid) {           // persistent CTAs drawing (signal, split) tasks from a ticket counter at the end of the workspace
            wa.n_tasks = (int)std::min<uint64_t>((uint64_t)wl.nsplit * n_sig, 0x7fffffffull);
            wa.ticket = reinterpret_cast<int*>(base + sig_bytes + out_bytes + part_bytes);
            e = cudaMemsetAsync(wa.ticket, 0, sizeof(int), stream);
            if (e != cudaSuccess) return cuda_fail(e, "Welch ticket");
            grid = dim3((unsigned)std::min<long long>(wa.n_tasks, (long long)eng->num_sms * std::max(1, bps)), 1);
        }
        e = cudaLaunchKernel(wk->fn, grid, dim3(wk->cta), wargs, wk->smem, stream);
        if (e != cudaSuccess) return cuda_fail(e, "launch welch_accum_kernel");
        eng->launches++;
        int n = (int)nfft, slots = wl.nsplit * wk->slots;
        void* fargs[] = { &wa, &n, &slots };
        e = cudaLaunchKernel(wk->fin, dim3((n + 255) / 256, n_sig), dim3(256), fargs, 0, stream);
        if (e != cudaSuccess) return cuda_fail(e, "launch welch_finalize_kernel");
        eng->launches++;
        char nm[96];
        snprintf(nm, sizeof(nm), "%s<%s,%d>", wk->mid ? "welch_accum_mid_kernel" : "welch_accum_kernel",
                 wl.prec == SA_PREC_F64 ? "double" : "float", wk->n);
        eng->last_kernel = nm;
    } else {
        const void* fn = wl.prec == SA_PREC_F64 ? (const void*)&psd_direct_kernel<double> : (const void*)&psd_direct_kernel<float>;
        int bps = 0;
        rc = eng->kernel_grid(fn, 256, 200 * 1024, &bps);                    // raises the dynamic shared memory limit once
        if (rc) return rc;
        int n = (int)nfft;
        void* dargs[] = { &wa, &n };
        e = cudaLaunchKernel(fn, dim3((nfft + 255) / 256, n_sig), dim3(256), dargs, wl.direct_smem, stream);
        if (e != cudaSuccess) return cuda_fail(e, "launch psd_direct_kernel");
        eng->launches++;
        eng->last_kernel = wl.prec == SA_PREC_F64 ? "psd_direct_kernel<double>" : "psd_direct_kernel<float>";
    }
    // rows -> their destinations (contiguous runs collapse into one copy)
    for (uint32_t i = 0; i < n_sig && e == cudaSuccess && !contiguous;) {
        uint32_t j = i + 1;
        while (j < n_sig && wl.d_out[j] == wl.d_out[j - 1] + nfft) j++;
        if (wl.d_out[i])
            e = cudaMemcpyAsync(wl.d_out[i], d_rows + (size_t)i * nfft, (size_t)(j - i) * nfft * sizeof(double),
                                cudaMemcpyDeviceToDevice, stream);
        i = j;
    }
    if (e != cudaSuccess) return cuda_fail(e, "PSD rows");
    return SA_OK;
}

// Runs the downconverter (and optionally the Welch PSD) for a batch on DEVICE samples.  d_out_iq == NULL: only the
// PSD rows are produced -- the decimated IQ then lives only in the FP32 scratch rows, which are reused batch after
// batch and stay in L2.  Batches of annotations alternate between the caller's stream and a helper stream so that
// the (issue-bound) Welch kernels of one batch overlap the (memory-bound) downconverter of the next.
static int run_batch_device(Engine* eng, const void* d_iq, uint64_t n_samples, int dtype, int big_endian,
                            double sample_rate, const sa_annotation* anns, uint32_t n_ann, uint32_t psd_nfft,
                            uint64_t psd_hop, int psd_window, double* d_out_iq, const uint64_t* iq_offsets,
                            double* d_out_psd, cudaStream_t stream) {
    const AnalysisProfile& pf = eng->profile;
    if (dtype == SA_DT_OTHER) dtype = SA_CF32;                                    // strict_reference: ExtractDownConvertService.java:93-96
    int dk = dtype_kind(dtype);
    if (pf.strict_reference && dtype == SA_CF64) dk = DK_CF64_S8;                 // :60-67,79-81
    const bool raw_wide = (dk == DK_CF64 || dk == DK_CF64_S8);
    static const char* pipe_env = getenv("SA_DC_PIPE");
    const bool pipe_ok = (pipe_env ? atoi(pipe_env) != 0 : true) && !raw_wide;
    std::vector<DcAnn> plan(n_ann);
    std::vector<float> taps;
    std::map<int, int> taps_off;
    std::vector<char> piped(n_ann, 0), rowsk(n_ann, 0);
    // row-per-thread kernel: 16-byte cp.async of raw rows, so a 16-byte aligned base and rows that start on a chunk boundary
    static const char* rows_env = getenv("SA_DC_ROWS");
    const bool rows_ok = (rows_env ? atoi(rows_env) != 0 : true) && (dk == DK_CF32 || dk == DK_CI16 || dk == DK_C8) && ((uintptr_t)d_iq & 15) == 0;
    const long long rows_spc = dk == DK_CF32 ? 2 : (dk == DK_CI16 ? 4 : 8);
    uint64_t scr_total = 0;
    for (uint32_t i = 0; i < n_ann; i++) {
        DcAnn& a = plan[i];
        const int D = anns[i].down;
        a.start_sample = (long long)anns[i].start_sample;
        a.count = (long long)anns[i].count;
        const double fr = anns[i].freq_off - std::floor(anns[i].freq_off);    // frac in [0,1)
        a.phase_step = (unsigned long long)std::ldexp((long double)fr, 64);   // exact 64-bit phase increment
        a.fast = anns[i].fast ? 1 : 0;
        a.m_out = (long long)dc_out_len(pf, anns[i].count, D, a.fast);
        a.out_off = iq_offsets ? (long long)iq_offsets[i] : 0;
        a.scr_off = 0;
        a.down = D;
        const int L = pf.taps.empty() ? 8 * D + 1 : (int)pf.taps.size();
        a.n_taps = L;
        a.in_off = a.fast ? 0 : (pf.delay_mode == SA_DELAY_SAME ? (L - 1) / 2 : pf.delay_mode == SA_DELAY_VALID ? L - 1 : 0);
        if (!taps_off.count(D)) {
            // block layout: [pad so that ht is 16-byte aligned][h[0..max(8D, L-1)] zero padded][ht[r*8+p] = h[D*p+r]]
            std::vector<double> h;
            profile_taps(pf, D, h);
            const size_t nat = std::max<size_t>(h.size(), 8 * (size_t)D + 1);
            h.resize(nat, 0.0);
            while ((taps.size() + nat) % 4) taps.push_back(0.f);
            taps_off[D] = (int)taps.size();
            for (double v : h) taps.push_back((float)v);
            for (int r = 0; r < D; r++) for (int p = 0; p < 8; p++) taps.push_back((float)h[(size_t)D * p + r]);
        }
        a.taps_off = taps_off[D];
        a.qmagic = D > 1 ? (unsigned)(((1ull << 32) + (unsigned long long)D - 1) / (unsigned long long)D) : 0u;
        const bool wide = (a.fast ? (D > kDcStage / 8) : (D > kDcMaxDown)) || (!a.fast && L > 8 * D + 1);
        size_t rows_smem = 0;
        if (wide) {
            a.nb = 0;                       // marks the warp-per-output kernel
        } else if (rows_ok && a.fast && D % rows_spc == 0 && (a.start_sample & (rows_spc - 1)) == 0 &&
                   dc_fast_smem_bytes((int)(D / rows_spc)) <= kDcFastSmemMax) {
            a.nb = kDcFastRows;              // box-car mode of the row-per-thread kernel: one output per row, no halo
            rowsk[i] = 1;
        } else if (rows_ok && !a.fast && dc_rows_aligned(a.start_sample + a.in_off, rows_spc) && !(big_endian && dc_rows_shape(dk, D).mode == 0) &&
                   dc_rows_kernel(dk, D, dc_rows_shape(dk, D), &rows_smem)) {
            a.nb = dc_rows_shape(dk, D).nt - 8;
            rowsk[i] = 1;
        } else if (pipe_ok && !a.fast && D <= 32) {
            // pipelined variant: the whole tile is one register batch (<= 17 x 256 staged samples)
            // blocks per tile: the staged samples fill the register batch (n_stage + D - 1 <= 17 x 256) and the tile
            // (staged samples + 8 partial sums per block) stays within a third of the SM's shared memory; a thread
            // takes several blocks when the decimation is small (D = 2: 256 -> 768 blocks per tile)
            const int by_batch = (kDcPipeLoads * kDcThreads - D) / D;
            const int by_smem = (int)((size_t)(74 * 1024 - dc_tap_smem_bytes(D) - 64) / (8 * (size_t)(D + 1) + 64));
            int nblk = std::max(8, std::min(by_batch, by_smem));
            if (nblk > kDcThreads) nblk -= nblk % kDcThreads;        // whole rounds of one block per thread
            a.nb = nblk - 7;
            piped[i] = 1;
        } else {
            const int nblk = std::max(8, std::min(kDcThreads, kDcStage / D));
            a.nb = a.fast ? nblk : nblk - 7;
        }
    }
    // ---- batches: annotations in caller order, cut where the FP32 rows of a batch reach the batch size
    const bool want_psd = d_out_psd != nullptr;
    // FP32 rows per batch.  Round 2 cut the rows at 128 MB (about the L2) and alternated the batches between two streams;
    // with the row-per-thread downconverter at the HBM rate one batch for the whole call is faster (C3, 262 MB of rows:
    // 1.198 ms as one batch, 1.215 ms as two, 1.25 ms at 64-112 MB), so the cut is 512 MB now.  SA_DC_BATCH_MB overrides.
    static const char* batch_env = getenv("SA_DC_BATCH_MB");
    const uint64_t batch_mb = batch_env && atoi(batch_env) > 0 ? (uint64_t)atoi(batch_env) : 512;
    const uint64_t scr_cap_elems = (batch_mb << 20) / sizeof(float2);
    std::vector<std::pair<uint32_t, uint32_t>> batches;
    {
        const uint32_t max_per_batch = 65535;                // annotations are grid.y of the launches
        uint32_t b0 = 0;
        uint64_t acc = 0;
        for (uint32_t i = 0; i < n_ann; i++) {
            if (i > b0 && ((want_psd && acc + (uint64_t)plan[i].m_out + 1 > scr_cap_elems) || i - b0 >= max_per_batch)) {
                batches.push_back({b0, i}); b0 = i; acc = 0;
            }
            plan[i].scr_off = (long long)acc;
            acc += ((uint64_t)plan[i].m_out + 1) & ~(uint64_t)1;       // rows start 16-byte aligned (128-bit loads of the Welch kernel)
            if (want_psd) scr_total = std::max(scr_total, acc);
        }
        batches.push_back({b0, n_ann});
    }
    const bool dual = want_psd && batches.size() > 1;
    int rc = SA_OK;
    if (want_psd) {
        rc = eng->ensure_scratch(8, (dual ? 2 : 1) * std::max<uint64_t>(scr_total, 1) * sizeof(float2));
        if (rc) return rc;
    }
    // annotation plan (device): batch by batch, inside a batch sorted by (kernel, fast, down) so that launches group
    std::vector<DcAnn> sorted;
    sorted.reserve(n_ann);
    std::vector<uint32_t> order;
    order.reserve(n_ann);
    auto key = [&](uint32_t i) { return std::make_tuple(plan[i].nb == 0 ? 2 : (rowsk[i] ? 3 : (piped[i] ? 0 : 1)), plan[i].fast, plan[i].down); };
    for (auto& b : batches) {
        std::vector<uint32_t> o;
        for (uint32_t i = b.first; i < b.second; i++) o.push_back(i);
        std::stable_sort(o.begin(), o.end(), [&](uint32_t x, uint32_t y) { return key(x) < key(y); });
        for (uint32_t i : o) { order.push_back(i); sorted.push_back(plan[i]); }
    }
    // Welch launches of every batch, prepared before anything is launched.  Transform length min(psd_nfft, M) per
    // annotation (AnalysisDialogController.java:303-307); rows shorter than psd_nfft are padded with NaN.
    std::vector<std::vector<WelchLaunch>> welch(batches.size());
    std::vector<std::vector<uint32_t>> short_rows(batches.size());
    size_t n_sigs_total = 0;
    if (want_psd) {
        for (size_t bi = 0; bi < batches.size(); bi++) {
            const int par = dual ? (int)(bi & 1) : 0;
            const float2* scr = (const float2*)eng->scratch[8] + (size_t)par * scr_total;
            std::map<uint32_t, std::vector<WelchJob>> by_n;
            for (uint32_t i = batches[bi].first; i < batches[bi].second; i++) {
                WelchJob j;
                j.re = nullptr; j.im = nullptr;
                j.f32 = scr + plan[i].scr_off;
                j.n = plan[i].m_out;
                j.fs = sample_rate / (double)plan[i].down;
                j.d_out = d_out_psd + (size_t)i * psd_nfft;
                const uint32_t nf = (uint32_t)std::min<long long>((long long)psd_nfft, plan[i].m_out);
                if (nf < psd_nfft) short_rows[bi].push_back(i);
                if (nf > 0) by_n[nf].push_back(j);
            }
            for (auto& kv : by_n) {
                const uint64_t hop = kv.first == psd_nfft ? psd_hop : std::max<uint64_t>(1, kv.first / 4);
                welch[bi].emplace_back();
                rc = welch_prepare(eng, kv.second, kv.first, hop, psd_window, welch[bi].back());
                if (rc) return rc;
                n_sigs_total += kv.second.size();
            }
        }
    }
    // ONE upload of everything the kernels read: annotation plan, taps, Welch plans -- from a pinned buffer, so that
    // the copy is asynchronous and nothing later in the launch sequence has to touch pageable memory
    const size_t ann_bytes = (sorted.size() * sizeof(DcAnn) + 255) & ~(size_t)255;
    const size_t taps_bytes = (taps.size() * sizeof(float) + 255) & ~(size_t)255;
    const size_t sig_bytes = (n_sigs_total * sizeof(WelchSig) + 255) & ~(size_t)255;
    const size_t plan_bytes = ann_bytes + taps_bytes + sig_bytes;
    rc = eng->ensure_scratch(0, plan_bytes);
    if (rc) return rc;
    cudaError_t e = cudaSuccess;
    if (eng->h_plan_cap < plan_bytes) {
        if (eng->h_plan) { cudaEventSynchronize(eng->plan_ev); cudaFreeHost(eng->h_plan); }
        eng->h_plan = nullptr; eng->h_plan_cap = 0;
        e = cudaHostAlloc(&eng->h_plan, plan_bytes + (plan_bytes >> 1), cudaHostAllocPortable);
        if (e != cudaSuccess) return cuda_fail(e, "cudaHostAlloc(plan)");
        eng->h_plan_cap = plan_bytes + (plan_bytes >> 1);
    }
    if (!eng->plan_ev) {
        e = cudaEventCreateWithFlags(&eng->plan_ev, cudaEventDisableTiming);
        if (e != cudaSuccess) return cuda_fail(e, "plan event");
    } else {
        e = cudaEventSynchronize(eng->plan_ev);                 // the previous call's upload has left the buffer
        if (e != cudaSuccess) return cuda_fail(e, "plan event wait");
    }
    char* hp = (char*)eng->h_plan;
    memcpy(hp, sorted.data(), sorted.size() * sizeof(DcAnn));
    memcpy(hp + ann_bytes, taps.data(), taps.size() * sizeof(float));
    {
        size_t off = ann_bytes + taps_bytes;
        for (auto& wb : welch) for (auto& wl : wb) { memcpy(hp + off, wl.sigs.data(), wl.sigs.size() * sizeof(WelchSig)); off += wl.sigs.size() * sizeof(WelchSig); }
    }
    DcAnn* d_anns = (DcAnn*)eng->scratch[0];
    float* d_taps = (float*)((char*)eng->scratch[0] + ann_bytes);
    const WelchSig* d_sigs = (const WelchSig*)((char*)eng->scratch[0] + ann_bytes + taps_bytes);
    e = cudaMemcpyAsync(eng->scratch[0], hp, plan_bytes, cudaMemcpyHostToDevice, stream);
    if (e == cudaSuccess) e = cudaEventRecord(eng->plan_ev, stream);
    if (e != cudaSuccess) return cuda_fail(e, "upload annotation plan");

    // Two schedules for more than one batch:
    //   alternate (default): batch b runs downconverter and Welch on stream b & 1;
    //   pipelined (SA_DC_SCHED=1): every downconverter launch on the caller's stream, every Welch launch on a HIGH-PRIORITY
    //     helper stream behind an event, so that Welch of batch b could share the SMs with the downconverter of batch b + 1
    //     (the one bound by memory, the other by issue slots; with SA_WELCH_CTA=256 the Welch CTAs are small enough to fit
    //     beside the downconverter's).  Measured on C3 (ms; rows = schedule / Welch CTA, columns = SA_DC_BATCH_MB 16 32 64 128):
    //       pipelined 256: 1.568 1.477 1.384 1.356     pipelined 512: 1.621 1.475 1.393 1.350
    //       alternate 256: 1.567 1.477 1.372 1.335     alternate 512: 1.592 1.485 1.399 1.331
    //     -- no gain from the overlap, and small batches lose to their launch tails: two 128 MB batches stay the default.
    static const char* sched_env = getenv("SA_DC_SCHED");
    const bool pipelined = dual && sched_env && atoi(sched_env) == 1;
    cudaStream_t st[2] = { stream, stream };
    if (dual) {
        if (!eng->dc_aux) {
            int lo = 0, hi = 0;
            e = cudaDeviceGetStreamPriorityRange(&lo, &hi);          // hi = numerically smallest = greatest priority
            if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&eng->dc_aux, cudaStreamNonBlocking, hi);
            for (int j = 0; j < 2 && e == cudaSuccess; j++) e = cudaEventCreateWithFlags(&eng->dc_ev[j], cudaEventDisableTiming);
            for (int j = 0; j < 4 && e == cudaSuccess; j++) e = cudaEventCreateWithFlags(&eng->dc_pipe_ev[j], cudaEventDisableTiming);
            if (e != cudaSuccess) return cuda_fail(e, "analysis helper stream");
        }
        st[1] = eng->dc_aux;
        e = cudaEventRecord(eng->dc_ev[0], stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(eng->dc_aux, eng->dc_ev[0], 0);
        if (e != cudaSuccess) return cuda_fail(e, "analysis fork");
    }

    DcArgs da;
    memset(&da, 0, sizeof(da));
    fill_load_params(da.lp, d_iq, dtype, big_endian);
    da.n_samples = (long long)n_samples;
    da.anns = d_anns;
    da.taps = d_taps;
    da.out = d_out_iq;
    DcTapParams tp;                      // copied into the launch by cudaLaunchKernel (kernel-parameter bank)
    tp.h_last = 0.f; tp.down = 0;
    void* args[] = { &da, &tp };
    const char* dc_name = "";            // family of the last downconverter launch (sa_last_kernel_name)
    bool any_welch = false;
    uint32_t pos = 0;                    // position in `sorted`
    size_t sig_pos = 0;                  // position in the uploaded WelchSig array
    for (size_t bi = 0; bi < batches.size(); bi++) {
        const int par = dual ? (int)(bi & 1) : 0;
        cudaStream_t s = pipelined ? stream : st[par];
        if (pipelined && bi >= 2) {          // the rows of parity `par` are rewritten: Welch of batch bi - 2 must have read them
            e = cudaStreamWaitEvent(stream, eng->dc_pipe_ev[2 + par], 0);
            if (e != cudaSuccess) return cuda_fail(e, "analysis pipeline wait");
        }
        const uint32_t bn = batches[bi].second - batches[bi].first;
        da.scratch = want_psd ? (float2*)eng->scratch[8] + (size_t)par * scr_total : nullptr;
        for (uint32_t g0 = pos; g0 < pos + bn;) {
            uint32_t g1 = g0 + 1;
            while (g1 < pos + bn && key(order[g1]) == key(order[g0])) g1++;
            const DcAnn& first = sorted[g0];
            da.ann_base = (int)g0;
            da.tiles_per_cta = 1;
            if (first.nb == 0) {              // warp-per-output kernel
                long long tiles = 0;
                for (uint32_t i = g0; i < g1; i++) tiles = std::max<long long>(tiles, (sorted[i].m_out + 7) / 8);
                if (tiles > 0) {
                    e = cudaLaunchKernel(dc_kernel(dk, 2), dim3((unsigned)tiles, g1 - g0), dim3(256), args, 0, s);
                    if (e != cudaSuccess) return cuda_fail(e, "launch downconvert_wide_kernel");
                    eng->launches++;
                    dc_name = "downconvert_wide_kernel";
                }
            } else if (rowsk[order[g0]] && first.fast) {     // row-per-thread kernel, box-car mode
                long long tiles = 0;
                for (uint32_t i = g0; i < g1; i++) tiles = std::max<long long>(tiles, (sorted[i].m_out + first.nb - 1) / first.nb);
                const size_t smem = (size_t)dc_fast_smem_bytes(first.down / (int)rows_spc);
                const void* fn = dc_rows_fast_kernel(dk);
                const long long group_tiles = tiles * (long long)(g1 - g0);
                da.tiles_per_cta = group_tiles >= 16LL * 16 * eng->num_sms ? 16 : 4;
                const long long ctas = (tiles + da.tiles_per_cta - 1) / da.tiles_per_cta;
                if (ctas > 0) {
                    size_t& have = eng->dc_smem_set[fn];
                    if (have < smem) {
                        e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                        if (e != cudaSuccess) return cuda_fail(e, "downconvert smem attribute");
                        have = smem;
                    }
                    e = cudaLaunchKernel(fn, dim3((unsigned)ctas, g1 - g0), dim3(kDcFastRows), args, smem, s);
                    if (e != cudaSuccess) return cuda_fail(e, "launch downconvert_rows_fast_kernel");
                    eng->launches++;
                    dc_name = "downconvert_rows_fast_kernel";
                }
            } else if (rowsk[order[g0]]) {     // row-per-thread kernel
                long long tiles = 0;
                for (uint32_t i = g0; i < g1; i++) tiles = std::max<long long>(tiles, (sorted[i].m_out + first.nb - 1) / first.nb);
                size_t smem = 0;
                const DcRowsShape rows_shape = dc_rows_shape(dk, first.down);
                const void* fn = dc_rows_kernel(dk, first.down, rows_shape, &smem);
                std::vector<float> rt;
                dc_rows_taps(taps.data() + first.taps_off, first.down, rt);
                void* rargs[] = { &da, rt.data() };
                static const char* te = getenv("SA_DC_ROWS_TILES");
                const long long group_tiles = tiles * (long long)(g1 - g0);
                da.tiles_per_cta = te && atoi(te) > 0 ? atoi(te) : (group_tiles >= 16LL * 16 * eng->num_sms ? 16 : 4);
                const long long ctas = (tiles + da.tiles_per_cta - 1) / da.tiles_per_cta;
                if (ctas > 0) {
                    size_t& have = eng->dc_smem_set[fn];
                    if (have < smem) {
                        e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                        if (e != cudaSuccess) return cuda_fail(e, "downconvert smem attribute");
                        have = smem;
                    }
                    e = cudaLaunchKernel(fn, dim3((unsigned)ctas, g1 - g0), dim3(rows_shape.nt), rargs, smem, s);
                    if (e != cudaSuccess) return cuda_fail(e, "launch downconvert_rows_kernel");
                    eng->launches++;
                    dc_name = "downconvert_rows_kernel";
                }
            } else {
                long long tiles = 0;
                for (uint32_t i = g0; i < g1; i++) tiles = std::max<long long>(tiles, (sorted[i].m_out + first.nb - 1) / first.nb);
                const int D = first.down;
                const bool pipe = piped[order[g0]] != 0;
                const bool ptaps = !first.fast && D <= kDcParamMaxDown;
                if (ptaps) {
                    const float* h = taps.data() + first.taps_off;
                    tp.h_last = h[8 * D];
                    tp.down = D;
                    memcpy(tp.ht, h + (std::max<size_t>((size_t)first.n_taps, 8 * (size_t)D + 1)), sizeof(float) * 8 * (size_t)D);
                }
                const size_t smem = dc_smem_bytes(D, first.nb, first.fast, pipe);
                const void* fn = dc_kernel(dk, pipe ? 3 : (ptaps ? 1 : 0));
                if (pipe) {
                    // consecutive tiles per CTA: 8, or 16 when the launch still fills the GPU many times over (C3: 1.544 ->
                    // 1.524 ms; 4 / 33 tiles per CTA measured slower); SA_DC_TILES overrides
                    static const char* te = getenv("SA_DC_TILES");
                    const long long group_tiles = tiles * (long long)(g1 - g0);
                    da.tiles_per_cta = te && atoi(te) > 0 ? atoi(te)
                                     : (group_tiles >= 16LL * 2 * kDcPipeTiles * eng->num_sms ? 2 * kDcPipeTiles : kDcPipeTiles);
                }
                const long long ctas = (tiles + da.tiles_per_cta - 1) / da.tiles_per_cta;
                if (ctas > 0) {
                    size_t& have = eng->dc_smem_set[fn];
                    if (have < smem) {            // raise the kernel's dynamic shared memory limit only when it grows
                        e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                        if (e != cudaSuccess) return cuda_fail(e, "downconvert smem attribute");
                        have = smem;
                    }
                    e = cudaLaunchKernel(fn, dim3((unsigned)ctas, g1 - g0), dim3(kDcThreads), args, smem, s);
                    if (e != cudaSuccess) return cuda_fail(e, "launch downconvert_kernel");
                    eng->launches++;
                    dc_name = pipe ? "downconvert_kernel(pipelined)" : "downconvert_kernel";
                }
            }
            g0 = g1;
        }
        pos += bn;
        if (pipelined) {                     // Welch of this batch: helper stream, behind the downconverter launches above
            e = cudaEventRecord(eng->dc_pipe_ev[par], stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(eng->dc_aux, eng->dc_pipe_ev[par], 0);
            if (e != cudaSuccess) return cuda_fail(e, "analysis pipeline fork");
            s = eng->dc_aux;
        }
        if (want_psd) {
            // NaN padding first (the short spectra are written over the row start)
            for (uint32_t i : short_rows[bi]) {
                e = cudaMemsetAsync(d_out_psd + (size_t)i * psd_nfft, 0xFF, (size_t)psd_nfft * sizeof(double), s);   // 0xFF..FF = NaN
                if (e != cudaSuccess) return cuda_fail(e, "PSD row padding");
            }
            for (auto& wl : welch[bi]) {
                rc = welch_launch(eng, wl, d_sigs + sig_pos, s, par);
                if (rc) return rc;
                if (!wl.sigs.empty()) any_welch = true;
                sig_pos += wl.sigs.size();
            }
        }
        if (pipelined) {
            e = cudaEventRecord(eng->dc_pipe_ev[2 + par], eng->dc_aux);
            if (e != cudaSuccess) return cuda_fail(e, "analysis pipeline record");
        }
    }
    eng->last_kernel = any_welch ? std::string(dc_name) + "+" + eng->last_kernel : std::string(dc_name);
    if (dual) {
        e = cudaEventRecord(eng->dc_ev[1], eng->dc_aux);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(stream, eng->dc_ev[1], 0);
        if (e != cudaSuccess) return cuda_fail(e, "analysis join");
    }
    return SA_OK;
}

}  // namespace sa


static int check_psd(uint32_t nfft, uint64_t* hop, int32_t window) {
    if (nfft == 0) return set_error(SA_ERR_INVALID_ARG, "psd nfft is 0");
    if (*hop == 0) *hop = std::max<uint32_t>(1, nfft / 4);           // 75 % overlap
    if (window < SA_WIN_RECT || window > SA_WIN_BLACKMAN_HARRIS) return set_error(SA_ERR_INVALID_ARG, "unknown window %d", window);
    return SA_OK;
}

// dtype as the downconverter sees it: with strict_reference a datatype without a decode branch is read as cf32
// (ExtractDownConvertService.java:93-96) and all non-integer types use an 8-byte stride (:60-67)
static int dc_dtype(const sa_engine* engine, int32_t dtype, uint64_t* bps) {
    if (dtype == SA_DT_OTHER || (dtype == SA_CF64 && engine->profile.strict_reference)) {
        if (!engine->profile.strict_reference) return set_error(SA_ERR_UNSUPPORTED, "datatype without a decode branch (strict_reference is off)");
        *bps = 8;
        return SA_OK;
    }
    *bps = (uint64_t)sa_bytes_per_iq(dtype);
    if (!*bps) return set_error(SA_ERR_INVALID_ARG, "unknown dtype %d", dtype);
    return SA_OK;
}

extern "C" {

int32_t sa_lowpass_taps(int32_t down, double* taps) {
    if (down < 1 || !taps) return set_error(SA_ERR_INVALID_ARG, "down < 1 or taps NULL");
    std::vector<double> h;
    lowpass_taps(down, h);
    memcpy(taps, h.data(), h.size() * sizeof(double));
    return SA_OK;
}

void sa_analysis_config_init(sa_analysis_config* c) {
    if (!c) return;
    memset(c, 0, sizeof(*c));
    c->struct_size = sizeof(*c);
    c->delay_mode = SA_DELAY_CAUSAL;
    c->length_mode = SA_LEN_FLOOR;
    c->psd_scaling = SA_PSD_DENSITY;
    c->psd_detrend = SA_DETREND_NONE;
    c->psd_precision = SA_PREC_F32;
}

int32_t sa_set_analysis_config(sa_engine* engine, const sa_analysis_config* c) {
    ENGINE_ENTER(engine);
    AnalysisProfile pf;
    if (c) {
        if (c->struct_size != sizeof(*c)) return set_error(SA_ERR_INVALID_ARG, "config.struct_size %u != %zu", c->struct_size, sizeof(*c));
        if (c->delay_mode < SA_DELAY_CAUSAL || c->delay_mode > SA_DELAY_VALID) return set_error(SA_ERR_INVALID_ARG, "unknown delay_mode %d", c->delay_mode);
        if (c->length_mode != SA_LEN_FLOOR && c->length_mode != SA_LEN_CEIL) return set_error(SA_ERR_INVALID_ARG, "unknown length_mode %d", c->length_mode);
        if (c->psd_scaling != SA_PSD_DENSITY && c->psd_scaling != SA_PSD_SPECTRUM) return set_error(SA_ERR_INVALID_ARG, "unknown psd_scaling %d", c->psd_scaling);
        if (c->psd_detrend != SA_DETREND_NONE && c->psd_detrend != SA_DETREND_CONSTANT) return set_error(SA_ERR_INVALID_ARG, "unknown psd_detrend %d", c->psd_detrend);
        if (c->psd_precision != SA_PREC_AUTO && c->psd_precision != SA_PREC_F32 && c->psd_precision != SA_PREC_F64)
            return set_error(SA_ERR_INVALID_ARG, "unknown psd_precision %d", c->psd_precision);
        if ((c->taps == nullptr) != (c->n_taps == 0)) return set_error(SA_ERR_INVALID_ARG, "taps / n_taps disagree");
        if (c->n_taps > (1u << 20)) return set_error(SA_ERR_UNSUPPORTED, "more than 2^20 taps");
        for (uint32_t i = 0; i < c->n_taps; i++)
            if (!std::isfinite(c->taps[i])) return set_error(SA_ERR_INVALID_ARG, "tap %u is not finite", i);
        if (c->taps) pf.taps.assign(c->taps, c->taps + c->n_taps);
        pf.delay_mode = c->delay_mode; pf.length_mode = c->length_mode;
        pf.psd_scaling = c->psd_scaling; pf.psd_detrend = c->psd_detrend;
        pf.psd_precision = c->psd_precision == SA_PREC_F64 ? SA_PREC_F64 : SA_PREC_F32;
        pf.strict_reference = c->strict_reference ? 1 : 0;
    }
    engine->profile = pf;
    return SA_OK;
}

int32_t sa_get_analysis_config(sa_engine* engine, sa_analysis_config* out) {
    ENGINE_ENTER(engine);
    if (!out) return set_error(SA_ERR_INVALID_ARG, "out is NULL");
    const AnalysisProfile& pf = engine->profile;
    sa_analysis_config_init(out);
    out->taps = pf.taps.empty() ? nullptr : pf.taps.data();       // engine-owned, valid until the next sa_set_analysis_config
    out->n_taps = (uint32_t)pf.taps.size();
    out->delay_mode = pf.delay_mode; out->length_mode = pf.length_mode;
    out->psd_scaling = pf.psd_scaling; out->psd_detrend = pf.psd_detrend;
    out->psd_precision = pf.psd_precision; out->strict_reference = pf.strict_reference;
    return SA_OK;
}

uint64_t sa_downconvert_length(sa_engine* engine, uint64_t count, int32_t down, int32_t fast) {
    if (!engine || down < 1) return 0;
    std::lock_guard<std::mutex> lock_(engine->mu);
    return dc_out_len(engine->profile, count, down, fast);
}

int32_t sa_downconvert_psd_batch_device(sa_engine* engine, const void* d_iq, uint64_t iq_bytes, int32_t dtype,
                                        int32_t big_endian, double sample_rate, const sa_annotation* anns,
                                        uint32_t n_ann, uint32_t psd_nfft, uint64_t psd_hop, int32_t psd_window,
                                        double* d_out_iq, const uint64_t* iq_offsets, double* d_out_psd_db,
                                        void* cuda_stream) {
    ENGINE_ENTER(engine);
    uint64_t bps = 0;
    int rc = dc_dtype(engine, dtype, &bps);
    if (rc) return rc;
    if (n_ann == 0) return SA_OK;
    if (!d_out_iq && !d_out_psd_db) return set_error(SA_ERR_INVALID_ARG, "both outputs are NULL");
    if (d_out_iq && !iq_offsets) return set_error(SA_ERR_INVALID_ARG, "iq_offsets is NULL");
    if ((uintptr_t)d_iq % bps) return set_error(SA_ERR_INVALID_ARG, "d_iq must be aligned to %llu bytes", (unsigned long long)bps);
    rc = validate_anns(anns, n_ann, iq_bytes / bps, (dtype == SA_CF64 && engine->profile.strict_reference) ? 1 : 0);
    if (rc) return rc;
    if (d_out_psd_db) { rc = check_psd(psd_nfft, &psd_hop, psd_window); if (rc) return rc; }
    return run_batch_device(engine, d_iq, iq_bytes / bps, dtype, big_endian, sample_rate, anns, n_ann, psd_nfft, psd_hop,
                            psd_window, d_out_iq, iq_offsets, d_out_psd_db, (cudaStream_t)cuda_stream);
}

int32_t sa_downconvert_psd_batch(sa_engine* engine, const void* iq, uint64_t iq_bytes, int32_t dtype, int32_t big_endian,
                                 double sample_rate, const sa_annotation* anns, uint32_t n_ann, uint32_t psd_nfft,
                                 uint64_t psd_hop, int32_t psd_window, double* out_iq, const uint64_t* iq_offsets,
                                 double* out_psd_db) {
    ENGINE_ENTER(engine);
    uint64_t bps = 0;
    int rc = dc_dtype(engine, dtype, &bps);
    if (rc) return rc;
    if (n_ann == 0) return SA_OK;
    if (!iq) return set_error(SA_ERR_INVALID_ARG, "iq is NULL");
    if (out_iq && !iq_offsets) return set_error(SA_ERR_INVALID_ARG, "iq_offsets is NULL");
    const uint64_t extra = (dtype == SA_CF64 && engine->profile.strict_reference) ? 1 : 0;   // the stride bug reads one double past the span
    rc = validate_anns(anns, n_ann, iq_bytes / bps, extra);
    if (rc) return rc;
    if (out_psd_db) { rc = check_psd(psd_nfft, &psd_hop, psd_window); if (rc) return rc; }

    // Only the annotated spans cross PCIe: each annotation's samples are copied into a packed
    // device buffer (16-byte aligned spans) and the plan is rebased onto it.
    Slot& s = engine->slots[0];
    std::vector<sa_annotation> local(anns, anns + n_ann);
    std::vector<uint64_t> dev_off(n_ann);
    const uint64_t align = 16 / std::min<uint64_t>(bps, 16);                       // samples per 16 bytes
    uint64_t in_samples = 0, out_doubles = 0;
    for (uint32_t i = 0; i < n_ann; i++) {
        local[i].start_sample = in_samples;
        in_samples += (anns[i].count + extra + align - 1) / align * align;
        dev_off[i] = out_doubles;
        out_doubles += 2 * dc_out_len(engine->profile, anns[i].count, anns[i].down, anns[i].fast);
    }
    const size_t psd_bytes = out_psd_db ? (size_t)n_ann * psd_nfft * sizeof(double) : 0;
    const size_t iq_out_bytes = out_iq ? (size_t)out_doubles * 8 : 0;
    rc = engine->ensure_slot(s, std::max<size_t>(in_samples * bps, 16), std::max<size_t>(iq_out_bytes + psd_bytes, 16));
    if (rc) return rc;
    cudaError_t e = cudaSuccess;
    if (host_ptr_is_pinned(iq)) {
        for (uint32_t i = 0; i < n_ann && e == cudaSuccess; i++) {
            if (anns[i].count)
                e = cudaMemcpyAsync((char*)s.d_in + local[i].start_sample * bps, (const char*)iq + anns[i].start_sample * bps,
                                    (anns[i].count + extra) * bps, cudaMemcpyHostToDevice, s.stream);
        }
    } else {
        // pageable capture (mmapped file): pieces of <= 32 MiB alternate between the pinned staging buffers of
        // slots 1 and 2; an event per buffer says when its previous H2D has drained
        const size_t piece = 32u << 20;
        Slot* st[2] = { &engine->slots[1], &engine->slots[2] };
        struct Events {                                      // destroyed on every exit path
            cudaEvent_t ev[2] = { nullptr, nullptr };
            ~Events() { for (auto x : ev) if (x) { cudaEventSynchronize(x); cudaEventDestroy(x); } }
        } evs;
        cudaEvent_t* ev = evs.ev;
        for (int k = 0; k < 2 && e == cudaSuccess; k++) {
            rc = engine->ensure_staging(*st[k], piece, 0);
            if (rc) return rc;
            e = cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming);
        }
        int k = 0;
        for (uint32_t i = 0; i < n_ann && e == cudaSuccess; i++) {
            const uint64_t total = (anns[i].count ? anns[i].count + extra : 0) * bps;
            for (uint64_t off = 0; off < total && e == cudaSuccess; off += piece, k ^= 1) {
                const size_t nb = (size_t)std::min<uint64_t>(piece, total - off);
                e = cudaEventSynchronize(ev[k]);                 // a never-recorded event is complete
                if (e != cudaSuccess) break;
                engine->host_copy(st[k]->h_in, (const char*)iq + anns[i].start_sample * bps + off, nb);
                e = cudaMemcpyAsync((char*)s.d_in + local[i].start_sample * bps + off, st[k]->h_in, nb, cudaMemcpyHostToDevice, s.stream);
                if (e == cudaSuccess) e = cudaEventRecord(ev[k], s.stream);
            }
        }
    }
    // on failure nothing of the caller's may still be in flight when this returns
    auto fail = [&](int code) { cudaStreamSynchronize(s.stream); if (engine->dc_aux) cudaStreamSynchronize(engine->dc_aux); return code; };
    if (e != cudaSuccess) return fail(cuda_fail(e, "H2D annotation spans"));
    double* d_iq_out = out_iq ? (double*)s.d_out : nullptr;
    double* d_psd = out_psd_db ? (double*)((char*)s.d_out + iq_out_bytes) : nullptr;
    if (!d_iq_out && !d_psd) return fail(set_error(SA_ERR_INVALID_ARG, "both outputs are NULL"));
    rc = run_batch_device(engine, s.d_in, in_samples, dtype, big_endian, sample_rate, local.data(), n_ann, psd_nfft,
                          psd_hop, psd_window, d_iq_out, dev_off.data(), d_psd, s.stream);
    if (rc) return fail(rc);
    if (out_iq) {
        for (uint32_t i = 0; i < n_ann && e == cudaSuccess; i++) {
            const uint64_t m2 = 2 * dc_out_len(engine->profile, anns[i].count, anns[i].down, anns[i].fast);
            if (m2) e = cudaMemcpyAsync(out_iq + iq_offsets[i], d_iq_out + dev_off[i], m2 * 8, cudaMemcpyDeviceToHost, s.stream);
        }
    }
    if (e == cudaSuccess && out_psd_db)
        e = cudaMemcpyAsync(out_psd_db, d_psd, psd_bytes, cudaMemcpyDeviceToHost, s.stream);
    if (e != cudaSuccess) return fail(cuda_fail(e, "D2H annotation results"));
    e = cudaStreamSynchronize(s.stream);
    if (e != cudaSuccess) return cuda_fail(e, "annotation batch");
    return SA_OK;
}

int32_t sa_downconvert(sa_engine* engine, const void* iq, uint64_t iq_bytes, int32_t dtype, int32_t big_endian,
                       uint64_t start_sample, uint64_t count, double freq_off, int32_t down, int32_t fast,
                       double* out_re, double* out_im, uint64_t* out_len) {
    if (!out_re || !out_im || !out_len) return set_error(SA_ERR_INVALID_ARG, "NULL output");
    if (down < 1) return set_error(SA_ERR_INVALID_ARG, "down %d < 1", down);
    if (!engine) return set_error(SA_ERR_INVALID_ARG, "engine is NULL");
    const uint64_t m = sa_downconvert_length(engine, count, down, fast);
    sa_annotation a;
    a.start_sample = start_sample; a.count = count; a.freq_off = freq_off; a.down = down; a.fast = fast;
    std::vector<double> tmp(std::max<uint64_t>(2 * m, 1));
    const uint64_t off = 0;
    int rc = sa_downconvert_psd_batch(engine, iq, iq_bytes, dtype, big_endian, 1.0, &a, 1, 0, 0, 0, tmp.data(), &off, nullptr);
    if (rc) return rc;
    memcpy(out_re, tmp.data(), m * 8);
    memcpy(out_im, tmp.data() + m, m * 8);
    *out_len = m;
    return SA_OK;
}

int32_t sa_psd_welch(sa_engine* engine, const double* re, const double* im, uint64_t n, double fs, uint32_t nfft,
                     uint64_t hop, int32_t window, double* out_freq, double* out_db) {
    ENGINE_ENTER(engine);
    if (!re || !im || !out_freq || !out_db) return set_error(SA_ERR_INVALID_ARG, "NULL buffer");
    int rc = check_psd(nfft, &hop, window);
    if (rc) return rc;
    if (n < nfft) return set_error(SA_ERR_INVALID_ARG, "signal (%llu samples) shorter than nfft %u", (unsigned long long)n, nfft);
    if (!(fs > 0.0)) return set_error(SA_ERR_INVALID_ARG, "fs must be > 0");
    // stage the FP64 rows as a one-annotation batch whose "decimated IQ" is the input itself
    Slot& s = engine->slots[0];
    rc = engine->ensure_slot(s, 16, (size_t)(2 * n + nfft) * 8);
    if (rc) return rc;
    double* d_rows = (double*)s.d_out;
    double* d_psd = d_rows + 2 * n;
    auto fail = [&](int code) { cudaStreamSynchronize(s.stream); return code; };     // the caller's rows may be in flight
    cudaError_t e = cudaMemcpyAsync(d_rows, re, n * 8, cudaMemcpyHostToDevice, s.stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_rows + n, im, n * 8, cudaMemcpyHostToDevice, s.stream);
    if (e != cudaSuccess) return fail(cuda_fail(e, "H2D psd rows"));
    std::vector<WelchJob> jobs(1);
    jobs[0].re = d_rows; jobs[0].im = d_rows + n; jobs[0].f32 = nullptr; jobs[0].n = (long long)n; jobs[0].fs = fs;
    jobs[0].d_out = d_psd;
    WelchLaunch wl;
    rc = welch_prepare(engine, jobs, nfft, hop, window, wl);
    if (rc) return fail(rc);
    rc = welch_launch(engine, wl, nullptr, s.stream, 0);
    if (rc) return fail(rc);
    e = cudaMemcpyAsync(out_db, d_psd, (size_t)nfft * 8, cudaMemcpyDeviceToHost, s.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s.stream);
    if (e != cudaSuccess) return fail(cuda_fail(e, "psd welch"));
    for (uint32_t k = 0; k < nfft; k++) out_freq[k] = ((double)k - (double)(nfft / 2)) * fs / (double)nfft;
    return SA_OK;
}

}  // extern "C"
