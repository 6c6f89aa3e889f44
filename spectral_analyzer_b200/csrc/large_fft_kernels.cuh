// large_fft_kernels.cuh -- four-step FFT for transforms that do not fit one SM's shared memory
// (FP32 nfft 32768 / 65536, FP64 nfft 16384 / 32768 / 65536; nfft slider range main-scene.fxml:129).
//
// N = N1*N2, n = N2*n1 + n2, k = k1 + N1*k2:
//   large_cols_kernel : per frame and per group of C columns n2: decode + window, N1-point FFT over n1
//                       (register/shared-memory FFT of fft_core.cuh, threads of a column spread over
//                       warps so that the C columns are the fast thread index -> coalesced loads),
//                       multiply by W_N^(n2*k1), write A[k1][n2] to an L2-sized workspace.
//   large_rows_kernel : per frame and per group of C rows k1: N2-point FFT over n2 (contiguous loads),
//                       |X| -> dB, transpose the C x N2 tile through shared memory so that consecutive
//                       threads store consecutive bins k = k1 + N1*k2, fft-shifted.
// Same arithmetic contract as spectrogram_kernel (SpectralService.java:33-85, MainController.java:980-999).
#pragma once
#include "spectrogram_tma_kernel.cuh"

#ifndef SA_LARGE_ROWS_MINB
#define SA_LARGE_ROWS_MINB 3
#endif
#ifndef SA_LARGE_COLS_MINB
#define SA_LARGE_COLS_MINB 3
#endif

namespace sa {

constexpr int kLargeC = 16;      // columns / rows per CTA

// Exchange-buffer stride between the columns of large_cols_kernel: the column is the fast thread index, so
// consecutive lanes hit the same offset of consecutive buffers; a stride of 16 bytes (mod 128) spreads them
// over the banks and keeps the 128-bit stores of pass 0 aligned (without it all 16 columns share a bank:
// 16-way conflicts).
template <typename T, int N1> struct ColStride {
    static constexpr int E = (int)sizeof(cpx<T>), M = 128 / E, STEP = 16 / E, BASE = Geo<T, N1>::SM_ELEMS;
    static constexpr int value = BASE + ((STEP - BASE % M) + M) % M;
};

struct LargeArgs {
    SpecArgs s;                  // s.twiddle: pair table of the N1-point plan; s.window: T[N]
    long long frame0;            // first frame of this chunk
    const void* tw2;             // pair table of the N2-point plan
    const void* tw_n;            // cpx<T>[N]: W_N^j
    void* ws;                    // cpx<T>[chunk frames][N1][N2]
};

// column group `cg` (C columns n2) of `frame`: writes A[k1][n2] of that frame to ws_frame
template <typename T, int N1, int N2, int DK, bool WIN>
__device__ __forceinline__ void large_cols_body(const LargeArgs& a, const long long frame, cpx<T>* __restrict__ ws,
                                                const int cg, unsigned char* smem_raw) {
    using G = Geo<T, N1>;
    constexpr int P = G::P, TPF = G::TPF, N = N1 * N2, C = kLargeC;
    const int fl = threadIdx.x % C, t = threadIdx.x / C;          // column is the fast index
    cpx<T>* sm = reinterpret_cast<cpx<T>*>(smem_raw) + (size_t)fl * ColStride<T, N1>::value;
    const long long s0 = a.s.start_sample + frame * a.s.hop;
    if (s0 + N > a.s.n_samples) return;                           // EOF frame (uniform): the rows step writes the fill row
    const int n2 = cg * C + fl;
    cpx<T> v[P];
    if (a.s.lp.swap) {
#pragma unroll
        for (int q = 0; q < P; q++) v[q] = Loader<T, DK>::template load<true>(a.s.lp, s0 + (long long)(t + TPF * q) * N2 + n2);
    } else {
#pragma unroll
        for (int q = 0; q < P; q++) v[q] = Loader<T, DK>::template load<false>(a.s.lp, s0 + (long long)(t + TPF * q) * N2 + n2);
    }
    if constexpr (WIN) {
        const T* w = reinterpret_cast<const T*>(a.s.window);
#pragma unroll
        for (int q = 0; q < P; q++) { const T wv = __ldg(&w[(t + TPF * q) * N2 + n2]); v[q].x *= wv; v[q].y *= wv; }
    }
    TwSeed<T> seed; seed.om = mk2<T>((T)1, (T)0); seed.oh = seed.om;
    fft_frame<T, N1, false, false, true>(v, t, sm, reinterpret_cast<const cpx<T>*>(a.s.twiddle), nullptr, seed);
    // four-step twiddle W_N^(n2 k1), k1 = t + TPF q: W_N^(n2 t) advanced by W_N^(n2 TPF) per q (two table reads
    // per thread instead of P scattered ones; re-seeded from the table every 8 steps)
    const cpx<T>* twn = reinterpret_cast<const cpx<T>*>(a.tw_n);
    const cpx<T> step = __ldg(&twn[(n2 * TPF) & (N - 1)]);
    cpx<T> w = __ldg(&twn[(n2 * t) & (N - 1)]);
#pragma unroll
    for (int q = 0; q < P; q++) {
        const int k1 = t + TPF * q;
        if (q > 0) {
            if ((q & 7) == 0) w = __ldg(&twn[(n2 * k1) & (N - 1)]);
            else w = mk2<T>(fma_t(-w.y, step.y, w.x * step.x), fma_t(w.y, step.x, w.x * step.y));
        }
        ws[(size_t)k1 * N2 + n2] = mk2<T>(fma_t(-w.y, v[q].y, w.x * v[q].x), fma_t(w.y, v[q].x, w.x * v[q].y));
    }
}

template <typename T, int N1, int N2, int DK, bool WIN>
__global__ void __launch_bounds__(kLargeC * Geo<T, N1>::TPF, sizeof(T) == 4 ? SA_LARGE_COLS_MINB : 2)
large_cols_kernel(const LargeArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    large_cols_body<T, N1, N2, DK, WIN>(a, a.frame0 + blockIdx.y, reinterpret_cast<cpx<T>*>(a.ws) + (size_t)blockIdx.y * (N1 * N2),
                                        blockIdx.x, smem_raw);
}

// 16-byte / 8-byte loads of the workspace that bypass L1: each element is read once, so caching it in L1 gains nothing
__device__ __forceinline__ float2  ld_cg(const float2* p)  { return __ldcg(p); }
__device__ __forceinline__ double2 ld_cg(const double2* p) { return __ldcg(p); }

// row group `rg` (C rows k1) of `frame`: N2-point FFTs of A[k1][.] from ws_frame, dB, fft-shifted store.
// POOL (spectrum traces, SpecArgs::trace_acc): the tile carries |X|^2 instead of dB and the transposed bins are reduced
// into the frame's accumulator cell -- a separate instantiation, so that the rows path runs the code it always ran.
template <typename T, int N1, int N2, bool POOL = false, bool LVL = false>
__device__ __forceinline__ void large_rows_body(const LargeArgs& a, const long long frame, const cpx<T>* __restrict__ ws_frame,
                                                const int rg, unsigned char* smem_raw, const double* ltab = nullptr) {
    using G = Geo<T, N2>;
    constexpr int P = G::P, TPF = G::TPF, N = N1 * N2, C = kLargeC, THREADS = C * TPF;
    const int t = threadIdx.x % TPF, fl = threadIdx.x / TPF;      // element is the fast index
    cpx<T>* sm = reinterpret_cast<cpx<T>*>(smem_raw) + (size_t)fl * G::SM_ELEMS;
    const long long s0 = a.s.start_sample + frame * a.s.hop;
    const bool readable = s0 + N <= a.s.n_samples;                // CTA-uniform, MainController.java:987
    const int k1 = rg * C + fl;
    T db[P];
    if (readable) {
        const cpx<T>* ws = ws_frame + (size_t)k1 * N2;
        cpx<T> v[P];
#pragma unroll
        for (int q = 0; q < P; q++) v[q] = ld_cg(&ws[t + TPF * q]);
        TwSeed<T> seed; seed.om = mk2<T>((T)1, (T)0); seed.oh = seed.om;
        fft_frame<T, N2, false, false, true>(v, t, sm, reinterpret_cast<const cpx<T>*>(a.tw2), nullptr, seed);
        if constexpr (POOL) {
#pragma unroll
            for (int q = 0; q < P; q++) db[q] = fma_t(v[q].x, v[q].x, v[q].y * v[q].y);
        } else {
            if (a.s.db_mode == DBM_MAG_1E10) bins_to_db<T, P, DBM_MAG_1E10>(v, db, ltab);
            else bins_to_db<T, P, DBM_POWER>(v, db, ltab);
        }
    } else {
#pragma unroll
        for (int q = 0; q < P; q++) db[q] = POOL ? (T)a.s.trace_eof : (T)a.s.eof_fill;
    }
    // transpose the [C rows k1][N2 bins k2] tile so that consecutive threads hold consecutive k = k1 + N1*k2
    T* tile = reinterpret_cast<T*>(smem_raw);
    __syncthreads();
#pragma unroll
    for (int q = 0; q < P; q++) tile[(t + TPF * q) * (C + 1) + fl] = db[q];
    __syncthreads();
    const int c = threadIdx.x % C, j0 = threadIdx.x / C;
    const int kbase = rg * C + c;
    if constexpr (POOL) {
        constexpr int PT = N2 / (THREADS / C);                    // bins per thread
        static_assert(PT * (THREADS / C) == N2, "whole tile columns per thread");
        trace_store<T, PT, N>(a.s, trace_cell(a.s, frame),
                              [&](int i) { return (kbase + N1 * (j0 + i * (THREADS / C)) + N / 2) & (N - 1); },
                              [&](int i) { return tile[(j0 + i * (THREADS / C)) * (C + 1) + c]; });
        return;
    }
    const size_t row = (size_t)frame * N;
    for (int k2 = j0; k2 < N2; k2 += THREADS / C) {
        const T val = tile[k2 * (C + 1) + c];
        const size_t o = row + (size_t)((kbase + N1 * k2 + N / 2) & (N - 1));     // SpectralService.java:78
        if constexpr (LVL) { reinterpret_cast<unsigned char*>(a.s.out)[o] = db_level(val, a.s); continue; }
        if (a.s.out_kind == OUT_F32_DB) reinterpret_cast<float*>(a.s.out)[o] = (float)val;
        else if (a.s.out_kind == OUT_F64_DB) reinterpret_cast<double*>(a.s.out)[o] = (double)val;
        else reinterpret_cast<uint32_t*>(a.s.out)[o] = colormap_rgba((float)val, a.s);
    }
}

template <typename T, int N1, int N2, bool POOL = false>
__global__ void __launch_bounds__(kLargeC * Geo<T, N2>::TPF, SA_LARGE_ROWS_MINB)
large_rows_kernel(const LargeArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const double* ltab = nullptr;
    if constexpr (sizeof(T) == 8 && SA_F64_FAST_DB && !POOL) {
        __shared__ double s_ltab[128];
        f64_ltab_init(s_ltab);
        ltab = s_ltab;
    }
    large_rows_body<T, N1, N2, POOL>(a, a.frame0 + blockIdx.y, reinterpret_cast<const cpx<T>*>(a.ws) + (size_t)blockIdx.y * (N1 * N2),
                               blockIdx.x, smem_raw, ltab);
}

// level rows (OUT_LEVEL8, persistence spectra): the rows kernel with the level store instead of the dB store
template <typename T, int N1, int N2>
__global__ void __launch_bounds__(kLargeC * Geo<T, N2>::TPF, SA_LARGE_ROWS_MINB)
large_rows_level_kernel(const LargeArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const double* ltab = nullptr;
    if constexpr (sizeof(T) == 8 && SA_F64_FAST_DB) {
        __shared__ double s_ltab[128];
        f64_ltab_init(s_ltab);
        ltab = s_ltab;
    }
    large_rows_body<T, N1, N2, false, true>(a, a.frame0 + blockIdx.y, reinterpret_cast<const cpx<T>*>(a.ws) + (size_t)blockIdx.y * (N1 * N2),
                                            blockIdx.x, smem_raw, ltab);
}

struct LargeKernelInfo {
    const void* fn_cols; const void* fn_rows;
    const void* fn_rows_pool;    // large_rows_kernel<.., POOL>: spectrum-trace reduction instead of rows
    const void* fn_rows_level;   // large_rows_level_kernel: OUT_LEVEL8 rows
    int prec, n, n1, n2, dk, win;
    int cta_cols, cta_rows;
    size_t smem_cols, smem_rows;
};

void register_large_kernel(const LargeKernelInfo& k);     // engine.cu

template <typename T, int N1, int N2, int DK, bool WIN>
LargeKernelInfo make_large_info(int prec) {
    LargeKernelInfo k;
    k.fn_cols = (const void*)&large_cols_kernel<T, N1, N2, DK, WIN>;
    k.fn_rows = (const void*)&large_rows_kernel<T, N1, N2>;
    k.fn_rows_pool = (const void*)&large_rows_kernel<T, N1, N2, true>;
    k.fn_rows_level = (const void*)&large_rows_level_kernel<T, N1, N2>;
    k.prec = prec; k.n = N1 * N2; k.n1 = N1; k.n2 = N2; k.dk = DK; k.win = WIN ? 1 : 0;
    k.cta_cols = kLargeC * Geo<T, N1>::TPF;
    k.cta_rows = kLargeC * Geo<T, N2>::TPF;
    k.smem_cols = (size_t)kLargeC * ColStride<T, N1>::value * sizeof(cpx<T>);
    const size_t ex = (size_t)kLargeC * Geo<T, N2>::SM_ELEMS * sizeof(cpx<T>);
    const size_t tile = (size_t)N2 * (kLargeC + 1) * sizeof(T);
    k.smem_rows = ex > tile ? ex : tile;
    return k;
}

}  // namespace sa
