// spectrogram_kernel.cuh -- decode -> frame -> window -> FFT -> |X| -> dB (-> RGBA) in one kernel.
//
// Replaces, for a whole batch of frames, the loop of S/controllers/MainController.java:980-999
// around S/services/SpectralService.java:33-85 (and, for SA_OUT_RGBA8, the per-pixel colour
// mapping of MainController.java:1273-1285 with getColorForMagnitude :926-957).
// Persistent CTAs walk frame blocks with a grid stride; every frame is read straight from global
// memory with coalesced per-point loads (thread t takes points t + TPF*q), transformed in
// registers/shared memory (fft_core.cuh) and written as one fft-shifted row.
#pragma once
#include "decode.cuh"

#ifndef SA_POOL_EPILOGUE
#define SA_POOL_EPILOGUE 1      // 0: compile the fused display pooling out of the epilogues (A/B of its cost on the row path)
#endif
#ifndef SA_STORE_STREAMING
#define SA_STORE_STREAMING 0
#endif

namespace sa {

// OUT_LEVEL8 (internal, persistence spectra, persistence.cu): one byte per bin, the level of the dB value the F32 / F64
// row would hold, level = quantize(dB) with SpecArgs::lvl_*.  Only the *_level_kernel instantiations (store_row /
// store_fill with LVL = true) write it, so the kernels of every other output compile to what they were.
enum { OUT_F32_DB = 0, OUT_F64_DB = 1, OUT_RGBA8 = 2, OUT_LEVEL8 = 3 };
enum { DBM_MAG_1E10 = 0, DBM_POWER = 1 };

struct SpecArgs {
    LoadParams  lp;
    long long   n_samples;     // IQ pairs readable from lp.base
    long long   start_sample;  // MainController.java:984 currentSampleOffset
    long long   hop;
    long long   n_frames;
    const void* window;        // T[N] or nullptr
    const void* twiddle;       // cpx<T>[Geo::TW_ELEMS]
    const void* aux;           // spectrogram_mid_kernel: cpx<T>[N] roots W_N^j
    void*       out;
    int         out_kind;
    int         db_mode;
    double      eof_fill;      // -150.0, MainController.java:996-997
    // renderSpectrogram parameters (RGBA8 only)
    float       cmap_bias;     // -(conv + min_db) * inv_range, conv = 10*log10(fs/N) + 20*log10(N) (:1273-1274)
    float       inv_range;     // 1/(max_db - min_db), :929
    int         cmap;
    // display pooling fused into the epilogue (sa_render_canvas with MAX / MEAN): instead of a dB row per frame, |X|^2 is
    // reduced over the pool_fpc frames of a canvas column into out = float[columns][N] (fft-shifted bins, zero-initialised)
    int         pool_mode;     // 0: rows; 1: max; 2: sum; 3: spectrum trace (POOL_TRACE)
    float       pool_eof;      // |X|^2 whose level is eof_fill (frames past the end of the buffer)
    long long   pool_fpc;      // frames per canvas column (per trace row)
    unsigned long long pool_magic;   // ceil(2^64 / pool_fpc) (0 for pool_fpc == 1): column = umul64hi(frame, magic), exact
                                     // for frame * pool_fpc < 2^64 -- no 64-bit division (F2I / I2F sequences) in the kernels
    // spectrum traces (sa_spectrum_trace, trace.cu): |X|^2 in the launch's precision T is reduced into up to three
    // accumulators T[cells][N] (fft-shifted bins, zero-initialised): [0] sum (red.add), [1] max and [2] min (red.max on
    // the bit pattern, resp. on its complement).  A cell holds at most trace_kc = min(F, kTraceCellFrames) frames of ONE
    // row: cell = row * trace_cpr + (f - row * F) / trace_kc, row = f / F, f = frame + trace_frame0.
    // OUT_LEVEL8 launches are never pooled: their quantizer shares the trace fields' space, so that the arguments of
    // every other launch keep their layout (and the kernels their register allocation).
    union {
        struct {
            void*       trace_acc[3];  // nullptr: statistic not wanted
            long long   trace_frame0;  // frame of the accumulator that this launch's frame 0 is (host-pipeline chunks)
            long long   trace_cpr;     // cells per row
            unsigned long long trace_cmagic; // ceil(2^64 / trace_kc) (0 for trace_kc == 1)
            double      trace_eof;     // |X|^2 of a frame past the end of the buffer (as pool_eof, FP64)
        };
        // OUT_LEVEL8: u = (dB - lvl_min) * lvl_scale in the launch's precision T (both rounded to T, each operation
        // rounded on its own), level = u >= 1 ? (int)min(u, lvl_top) : 0 (below the range and NaN: 0, above: lvl_top)
        struct {
            double      lvl_min;
            double      lvl_scale;     // n_levels / (max_db - min_db)
            double      lvl_top;       // n_levels - 1
        };
    };
};
enum { POOL_TRACE = 3 };
constexpr int kTraceCellFrames = 256;       // frames per accumulator cell at most: an FP32 cell sums <= 256 terms
__device__ __forceinline__ long long pool_column(const SpecArgs& a, long long frame) {
    return a.pool_magic ? (long long)__umul64hi((unsigned long long)frame, a.pool_magic) : frame;
}
// accumulator cell of a frame: per frame, not per bin (two multiply-highs)
__device__ __forceinline__ long long trace_cell(const SpecArgs& a, long long frame) {
    const long long f = frame + a.trace_frame0;
    const long long row = pool_column(a, f);
    const unsigned long long r = (unsigned long long)(f - row * a.pool_fpc);
    return row * a.trace_cpr + (long long)(a.trace_cmagic ? __umul64hi(r, a.trace_cmagic) : r);
}

// One reduction per bin and frame, 32 consecutive bins per warp instruction: the L2 atomic units see one 128-byte line
// per instruction, the same number of transactions as the row stores they replace, and the accumulator (columns x N
// floats, a few MB) never leaves L2.  |X|^2 >= 0, so the unsigned order of the bit patterns is the float order.
__device__ __forceinline__ void pool_red(float* p, float v, int mode) {
    if (mode == 1) asm volatile("red.global.max.u32 [%0], %1;" ::"l"(p), "r"(__float_as_uint(v)) : "memory");
    else asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// Trace reductions, statistic S (0 sum, 1 max, 2 min) in the launch's precision.  MIN keeps the zero-initialised
// accumulator: the complement of the bit pattern reverses the order of non-negative values, so red.max of ~bits is
// the minimum, and an untouched cell (0) never wins.
template <int S> __device__ __forceinline__ void trace_red(float* p, float v) {
    if constexpr (S == 0) asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
    else asm volatile("red.global.max.u32 [%0], %1;" ::"l"(p), "r"(S == 1 ? __float_as_uint(v) : ~__float_as_uint(v)) : "memory");
}
template <int S> __device__ __forceinline__ void trace_red(double* p, double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    if constexpr (S == 0) asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
    else asm volatile("red.global.max.u64 [%0], %1;" ::"l"(p), "l"(S == 1 ? b : ~b) : "memory");
}
// one reduction per wanted statistic, bin and frame: bin idx(q) of cell `cell` takes pw(q), q < P (the power is
// recomputed per statistic rather than held in P more registers)
template <typename T, int P, int N, typename Idx, typename Pw>
__device__ __forceinline__ void trace_store(const SpecArgs& a, const long long cell, Idx idx, Pw pw) {
#pragma unroll
    for (int s = 0; s < 3; s++) {
        if (!a.trace_acc[s]) continue;                 // uniform
        T* o = reinterpret_cast<T*>(a.trace_acc[s]) + (size_t)cell * N;
#pragma unroll
        for (int q = 0; q < P; q++) {
            if (s == 0) trace_red<0>(&o[idx(q)], (T)pw(q));
            else if (s == 1) trace_red<1>(&o[idx(q)], (T)pw(q));
            else trace_red<2>(&o[idx(q)], (T)pw(q));
        }
    }
}

// level of a dB value (SpecArgs::lvl_*), exactly as include/sa_engine.h defines it for sa_spectrum_persistence.
// (int)c of c in [1, 255] is the low mantissa byte of c + 2^23 (2^52) added toward zero: no F2I, the FMA pipe only.
__device__ __forceinline__ unsigned char db_level(float d, const SpecArgs& a) {
    const float u = __fmul_rn(__fsub_rn(d, (float)a.lvl_min), (float)a.lvl_scale);
    const unsigned int b = __float_as_uint(__fadd_rz(fminf(u, (float)a.lvl_top), 8388608.0f));
    return u >= 1.0f ? (unsigned char)b : 0;
}
__device__ __forceinline__ unsigned char db_level(double d, const SpecArgs& a) {
    const double u = __dmul_rn(__dsub_rn(d, a.lvl_min), a.lvl_scale);
    const unsigned int b = (unsigned int)__double2loint(__dadd_rz(fmin(u, a.lvl_top), 4503599627370496.0));
    return u >= 1.0 ? (unsigned char)b : 0;
}

#ifndef SA_F64_FAST_DB
#define SA_F64_FAST_DB 1        // table-driven FP64 dB epilogue (0: library log10 / sqrt)
#endif
__device__ __forceinline__ float lg2_approx(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float sqrt_approx(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// SpectralService.java:80-81: 20*log10(abs + 1e-10)
template <int MODE> __device__ __forceinline__ float to_db(float re, float im) {
    const float p = __fmaf_rn(re, re, im * im);
    if constexpr (MODE == DBM_MAG_1E10) return 6.02059991327962f * lg2_approx(sqrt_approx(p) + 1e-10f);
    return 3.01029995663981f * lg2_approx(p + 1e-20f);
}
template <int MODE> __device__ __forceinline__ double to_db(double re, double im) {
    if constexpr (MODE == DBM_MAG_1E10) return 20.0 * log10(sqrt(re * re + im * im) + 1e-10);
    return 10.0 * log10(re * re + im * im + 1e-20);
}

// ---- FP64 dB without the library log10 / sqrt ----
// The literal form costs ~100 of the ~160 instructions per bin of the FP64 kernels.  Within the FP64 tolerance of
// 1e-9 dB:  20 log10(|X| + c) = 10 log10 p + 20 log10(1 + c / |X|),  p = |X|^2;  for p >= 1e-10 the second term is
// (20 / ln 10) (eps - eps^2 / 2), eps = c rsqrt(p) <= 1e-5, evaluated in FP32 (< 3e-11 dB);  log2 p = e + log2 m,
// m in [1, 2) split by its top 7 mantissa bits k: m c_k = 1 + r, c_k = rcp.approx(cell midpoint) (one MUFU, the same
// value the table was built from), |r| <= 2^-8, log1p(r) to r^4 / 4 (truncation 2e-13), -log2 c_k from a 128-entry
// shared-memory table filled at kernel start with the library log2.  Bins below the threshold (or non-finite) take
// the literal form, per thread.
__device__ __forceinline__ float rcp_approx(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rsqrt_approx(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float ltab_cell_mid(int k) { return __int_as_float(0x3f800000 | (k << 16) | 0x8000); }   // 1 + (k + 0.5) / 128
__device__ __forceinline__ void f64_ltab_init(double* tab) {          // every thread of the CTA, before the first frame
    for (int k = threadIdx.x; k < 128; k += blockDim.x) tab[k] = -log2((double)rcp_approx(ltab_cell_mid(k)));
    __syncthreads();
}
__device__ __forceinline__ double log2_tab(const double p, const double* tab) {      // p normal, positive
    const int hi = __double2hiint(p);
    const int k = (hi >> 13) & 127;
    const double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(p));
    const double r = fma(m, (double)rcp_approx(ltab_cell_mid(k)), -1.0);
    double q = fma(r, -0.25, 1.0 / 3.0);
    q = fma(r, q, -0.5);
    q = fma(r, q, 1.0);                                    // log1p(r) / r
    const double e = (double)((hi >> 20) - 1023);
    return fma(r * q, 1.4426950408889634074, e + tab[k]);
}

// dB of all P bins of a thread.  FP32 fast path for MAG_1E10: when |X| >= 2^-9 the FP32 sum
// |X| + 1e-10 rounds back to |X| (ulp(|X|) >= 2^-32, so 1e-10 is below half an ulp), hence
// 20 log10(|X| + 1e-10) equals 10 log10(|X|^2) and the square root is skipped; threads holding a
// bin with |X|^2 < 2^-18 take the literal form.
template <typename T, int P, int MODE>
__device__ __forceinline__ void bins_to_db(const cpx<T> (&v)[P], T (&db)[P], const double* tab = nullptr) {
    if constexpr (sizeof(T) == 4 && MODE == DBM_MAG_1E10) {
        // |X|^2 and the dB scale run two bins per issue slot (FMUL2 / FFMA2)
        float pmin = 3.0e38f;
#pragma unroll
        for (int q = 0; q < P; q += 2) {
            const pk2 xr = pack2(v[q].x, v[q + 1].x), xi = pack2(v[q].y, v[q + 1].y);
            unpack2(fma2(xr, xr, mul2(xi, xi)), db[q], db[q + 1]);
            pmin = fminf(pmin, fminf(db[q], db[q + 1]));
        }
        if (pmin >= 3.814697265625e-6f) {      // 2^-18
#pragma unroll
            for (int q = 0; q < P; q += 2)
                unpack2(mul2(pack2(lg2_approx(db[q]), lg2_approx(db[q + 1])), bcast2(3.01029995663981f)), db[q], db[q + 1]);
        } else {
#pragma unroll
            for (int q = 0; q < P; q++) db[q] = 6.02059991327962f * lg2_approx(sqrt_approx(db[q]) + 1e-10f);
        }
    } else if constexpr (sizeof(T) == 8 && SA_F64_FAST_DB) {
        bool fast = true;
#pragma unroll
        for (int q = 0; q < P; q++) {
            db[q] = fma(v[q].x, v[q].x, v[q].y * v[q].y);
            if constexpr (MODE == DBM_MAG_1E10) fast = fast && (db[q] >= 1e-10) && (db[q] < 1e300);
            else fast = fast && (db[q] < 1e300);           // p + 1e-20 is always a normal number; NaN fails
        }
        if (fast) {
#pragma unroll
            for (int q = 0; q < P; q++) {
                if constexpr (MODE == DBM_MAG_1E10) {
                    const float eps = 1e-10f * rsqrt_approx((float)db[q]);
                    const float corr = 8.685889638065037f * eps * __fmaf_rn(-0.5f, eps, 1.0f);
                    db[q] = fma(log2_tab(db[q], tab), 3.0102999566398119521, (double)corr);
                } else {
                    db[q] = 3.0102999566398119521 * log2_tab(db[q] + 1e-20, tab);
                }
            }
        } else {
#pragma unroll
            for (int q = 0; q < P; q++) db[q] = to_db<MODE>(v[q].x, v[q].y);
        }
    } else {
#pragma unroll
        for (int q = 0; q < P; q++) db[q] = to_db<MODE>(v[q].x, v[q].y);
    }
}

// getColorForMagnitude (MainController.java:926-957) on float components, channels packed
// R | G<<8 | B<<16 | A<<24.  n = clamp((dB - conv - min)/(max - min), 0, 1) is one saturating FMA
// (cmap_bias = -(conv + min_db) * inv_range, NaN -> 0); the Heatmap ramps are saturating FMAs too:
//   r = sat((n - 0.2)/0.3)   (0 below 0.2, the BLUE->RED ramp, 1 from 0.5 on)
//   g = sat(2 n - 1)         (0 below 0.5, the RED->YELLOW ramp)
//   b = n >= 0.2 ? 1 - r : 0
// and round(c * 255) is the low mantissa byte of c * 255 + 1.5 * 2^23 (no F2I).
template <int HEAT>
__device__ __forceinline__ uint32_t colormap_px(const float db, const float scale, const float bias) {
    const float n = __saturatef(__fmaf_rn(db, scale, bias));
    constexpr float MAGIC = 12582912.0f;
    if constexpr (HEAT) {
        const float r = __saturatef(__fmaf_rn(n, 1.0f / 0.3f, -0.2f / 0.3f));
        const float g = __saturatef(__fmaf_rn(n, 2.0f, -1.0f));
        const uint32_t R = __float_as_uint(__fmaf_rn(r, 255.0f, MAGIC));
        const uint32_t G = __float_as_uint(__fmaf_rn(g, 255.0f, MAGIC));
        // b = n >= 0.2 ? 1 - r : 0, scaled: 255 (1 - r) + magic; the blue magic carries alpha in mantissa bits 8..15
        constexpr float MAGIC_A = MAGIC + 65280.0f;
        const uint32_t B = __float_as_uint(n >= 0.2f ? __fmaf_rn(r, -255.0f, MAGIC_A + 255.0f) : MAGIC_A);
        const uint32_t rg = __byte_perm(R, G, 0x0040);          // byte0 = R, byte1 = G
        return __byte_perm(rg, B, 0x5410);                      // byte2 = B, byte3 = alpha (byte 1 of B's magic)
    } else {
        const uint32_t V = __float_as_uint(__fmaf_rn(n, 255.0f, MAGIC));
        return __byte_perm(V, 0xFF000000u, 0x7000);             // R = G = B = V, A = 255
    }
}
__device__ __forceinline__ uint32_t colormap_rgba(float db, const SpecArgs& a) {
    return a.cmap == 1 ? colormap_px<1>(db, a.inv_range, a.cmap_bias) : colormap_px<0>(db, a.inv_range, a.cmap_bias);
}

template <int DK> __host__ __device__ constexpr int bytes_per_iq_kind() {
    return DK == DK_CF32 ? 8 : DK == DK_CI16 ? 4 : DK == DK_C8 ? 2 : 16;
}

// EOF row: frames that would read past the end of the buffer (MainController.java:994-998)
template <typename T, int N, bool LVL = false>
__device__ __forceinline__ void store_fill(const SpecArgs& a, const long long frame, const int t) {
    constexpr int P = Geo<T, N>::P, TPF = Geo<T, N>::TPF;
    if (SA_POOL_EPILOGUE && a.pool_mode) {
        if (a.pool_mode == POOL_TRACE) {
            const T pe = (T)a.trace_eof;
            trace_store<T, P, N>(a, trace_cell(a, frame), [&](int q) { return t + TPF * q; }, [&](int) { return pe; });
            return;
        }
        float* o = reinterpret_cast<float*>(a.out) + (size_t)pool_column(a, frame) * N;
#pragma unroll
        for (int q = 0; q < P; q++) pool_red(&o[t + TPF * q], a.pool_eof, a.pool_mode);
        return;
    }
    const size_t row = (size_t)frame * N;
    if (a.out_kind == OUT_F32_DB) {
        float* o = reinterpret_cast<float*>(a.out) + row;
#pragma unroll
        for (int q = 0; q < P; q++) o[t + TPF * q] = (float)a.eof_fill;
    } else if (a.out_kind == OUT_F64_DB) {
        double* o = reinterpret_cast<double*>(a.out) + row;
#pragma unroll
        for (int q = 0; q < P; q++) o[t + TPF * q] = a.eof_fill;
    } else if (LVL && a.out_kind == OUT_LEVEL8) {
        unsigned char* o = reinterpret_cast<unsigned char*>(a.out) + row;
        const unsigned char lv = db_level((T)a.eof_fill, a);
#pragma unroll
        for (int q = 0; q < P; q++) o[t + TPF * q] = lv;
    } else {
        uint32_t* o = reinterpret_cast<uint32_t*>(a.out) + row;
        const uint32_t px = colormap_rgba((float)a.eof_fill, a);
#pragma unroll
        for (int q = 0; q < P; q++) o[t + TPF * q] = px;
    }
}

// Copies the twiddle table into shared memory (plans with Geo::TW_SMEM) and returns the pointer the
// passes read; the caller must __syncthreads() (setup_window does) or sync before first use.
template <typename T, int N>
__device__ __forceinline__ const cpx<T>* setup_twiddles(const SpecArgs& a, unsigned char* smem_raw) {
    using G = Geo<T, N>;
    const cpx<T>* tw = reinterpret_cast<const cpx<T>*>(a.twiddle);
    if constexpr (G::TW_SMEM) {
        cpx<T>* tsm = reinterpret_cast<cpx<T>*>(smem_raw + G::SMEM_BYTES);
        for (int i = threadIdx.x; i < (int)(G::TW_BYTES / sizeof(cpx<T>)); i += G::CTA) tsm[i] = __ldg(&tw[i]);
        __syncthreads();
        return tsm;
    } else {
        return tw;
    }
}

// Window factors in pair order (element m, element m + P/2), m = 0..P/2-1, as the first butterfly
// stage consumes them: a padded row per thread in shared memory (one 8/16-byte load per butterfly),
// or registers for the wide plans.  Returns the calling thread's row.
template <typename T, int N>
__device__ __forceinline__ const T* setup_window(const SpecArgs& a, unsigned char* wsm_raw,
                                                 T (&win_reg)[Geo<T, N>::WIN_SMEM ? 1 : Geo<T, N>::P], const int t) {
    using G = Geo<T, N>;
    constexpr int P = G::P, TPF = G::TPF;
    const T* w = reinterpret_cast<const T*>(a.window);
    if constexpr (G::WIN_SMEM) {
        T* wsm = reinterpret_cast<T*>(wsm_raw);
        for (int i = threadIdx.x; i < TPF * P; i += G::CTA) {
            const int tt = i % TPF, e = i / TPF;             // element e of thread tt: sample tt + TPF*e
            const int slot = e < P / 2 ? 2 * e : 2 * (e - P / 2) + 1;
            wsm[tt * G::WROW + slot] = __ldg(&w[i]);
        }
        __syncthreads();
        return wsm + t * G::WROW;
    } else {
#pragma unroll
        for (int m = 0; m < P / 2; m++) {
            win_reg[2 * m] = __ldg(&w[t + TPF * m]);
            win_reg[2 * m + 1] = __ldg(&w[t + TPF * (m + P / 2)]);
        }
        return win_reg;
    }
}

// Epilogue of one frame: |X| -> dB (-> colour), written as the fft-shifted row
// out[(k + N/2) % N] (SpectralService.java:76-82), k = t + TPF*q.
template <typename T, int N, bool LVL = false>
__device__ __forceinline__ void store_row(const SpecArgs& a, const long long frame, const int t,
                                          const cpx<T> (&v)[Plan<T, N>::P], const double* ltab = nullptr) {
    constexpr int P = Geo<T, N>::P, TPF = Geo<T, N>::TPF;
    if (SA_POOL_EPILOGUE && a.pool_mode) {          // |X|^2 only: the logarithm is taken once per pixel by canvas_power_kernel
        const int kp = (t + N / 2) & (N - 1);
        if (a.pool_mode == POOL_TRACE) {            // ... or once per trace bin by trace_finalize_kernel
            trace_store<T, P, N>(a, trace_cell(a, frame), [&](int q) { return (kp + TPF * q) & (N - 1); },
                                 [&](int q) { return fma_t(v[q].x, v[q].x, v[q].y * v[q].y); });
            return;
        }
        float* o = reinterpret_cast<float*>(a.out) + (size_t)pool_column(a, frame) * N;
#pragma unroll
        for (int q = 0; q < P; q++)
            pool_red(&o[(kp + TPF * q) & (N - 1)], (float)fma_t(v[q].x, v[q].x, v[q].y * v[q].y), a.pool_mode);
        return;
    }
    T db[P];
    if (a.db_mode == DBM_MAG_1E10) bins_to_db<T, P, DBM_MAG_1E10>(v, db, ltab);
    else bins_to_db<T, P, DBM_POWER>(v, db, ltab);
    const size_t row = (size_t)frame * N;
    const int k0 = (t + N / 2) & (N - 1);
    if (a.out_kind == OUT_F32_DB) {
        float* o = reinterpret_cast<float*>(a.out) + row;
#pragma unroll
        for (int q = 0; q < P; q++) {
#if SA_STORE_STREAMING
            __stcs(&o[(k0 + TPF * q) & (N - 1)], (float)db[q]);      // rows are never re-read: evict-first in L2
#else
            o[(k0 + TPF * q) & (N - 1)] = (float)db[q];
#endif
        }
    } else if (a.out_kind == OUT_F64_DB) {
        double* o = reinterpret_cast<double*>(a.out) + row;
#pragma unroll
        for (int q = 0; q < P; q++) o[(k0 + TPF * q) & (N - 1)] = (double)db[q];
    } else if (LVL && a.out_kind == OUT_LEVEL8) {        // the byte comes from the db[] the F32 / F64 row would store
        unsigned char* o = reinterpret_cast<unsigned char*>(a.out) + row;
#pragma unroll
        for (int q = 0; q < P; q++) o[(k0 + TPF * q) & (N - 1)] = db_level(db[q], a);
    } else {
        uint32_t* o = reinterpret_cast<uint32_t*>(a.out) + row;
        const float sc = a.inv_range, bi = a.cmap_bias;
        if (a.cmap == 1) {
#pragma unroll
            for (int q = 0; q < P; q++) o[(k0 + TPF * q) & (N - 1)] = colormap_px<1>((float)db[q], sc, bi);
        } else {
#pragma unroll
            for (int q = 0; q < P; q++) o[(k0 + TPF * q) & (N - 1)] = colormap_px<0>((float)db[q], sc, bi);
        }
    }
}

#define SA_KERNEL_NAME spectrogram_kernel
#define SA_KERNEL_LVL false
#include "spectrogram_kernel_body.inc"
// level rows (OUT_LEVEL8, persistence spectra)
#define SA_KERNEL_NAME spectrogram_level_kernel
#define SA_KERNEL_LVL true
#include "spectrogram_kernel_body.inc"

// ---- registry ----
struct SpecKernelInfo {
    const void* fn;
    const void* fn_level;   // the same kernel writing OUT_LEVEL8 rows (nullptr: none)
    int prec;       // 1 f32, 2 f64 (SA_PREC_*)
    int n;
    int dk;
    int win;
    int cta;
    int fpc;
    int minb;
    size_t smem;
    int p;          // points per thread
    int np;         // passes
    int radix[4];
    int tma;        // 1: TMA-staged variant (needs 16-byte aligned frames)
};

void register_spec_kernel(const SpecKernelInfo& k);   // engine.cu

template <typename T, int N, int DK, bool WIN>
SpecKernelInfo make_spec_info(int prec) {
    using G = Geo<T, N>;
    using PL = Plan<T, N>;
    SpecKernelInfo k;
    k.fn = (const void*)&spectrogram_kernel<T, N, DK, WIN>;
    k.fn_level = (const void*)&spectrogram_level_kernel<T, N, DK, WIN>;
    k.prec = prec; k.n = N; k.dk = DK; k.win = WIN ? 1 : 0;
    k.cta = G::CTA; k.fpc = G::FPC; k.minb = G::MINB; k.smem = G::SMEM_BYTES + G::TW_BYTES + (WIN ? G::WIN_BYTES : 0);
    k.p = G::P; k.np = PL::NP; k.tma = 0;
    for (int i = 0; i < 4; i++) k.radix[i] = PL::radix(i);
    return k;
}

}  // namespace sa
