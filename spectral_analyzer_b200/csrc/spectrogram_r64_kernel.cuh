// spectrogram_r64_kernel.cuh -- 4096-point FP32 spectrogram as TWO radix-64 passes.
//
// Same arithmetic contract and output as spectrogram_kernel (SpectralService.java:33-85 in the frame loop of
// MainController.java:980-999).  64 points per thread, 64 threads (two warps) per frame: the frame crosses
// shared memory ONCE (the 3-pass kernels of spectrogram_mid_kernel.cuh are bound by shared-memory wavefronts),
// at the price of 128 data registers per thread, i.e. 8 warps per SM.  The raw frame is staged by TMA
// (cp.async.bulk + mbarrier) into the frame's exchange buffer while pass 1 and the epilogue of the previous
// frame run, as in spectrogram_tma_kernel.cuh, because 8 warps cannot hide a global-load latency.
//   pass 0  radix 64 on v[q] = x[t + 64 q], window folded into the first stage; exchange write j*64 + m -> 65 t + m
//   pass 1  radix 64, twiddle W_4096^(t m) by the packed register recurrence, re-seeded half way
// Requires 16-byte aligned frames (same condition as the other staged kernels).  Measured against the 3-pass kernel
// (2^28..2^30 samples, hop 4096): cf32 0.898 -> 0.583 ms (55 % -> 85 % of the HBM roofline), ci16 1.29 -> 1.22 ms,
// cu8 2.22 -> 2.49 ms (the strided 2-byte reads of the staged frame cost more than the 128-bit loads of the 3-pass
// kernel), so it is built and used for cf32 and ci16 input only.
#pragma once
#include "spectrogram_tma_kernel.cuh"

#ifndef SA_CTA_R64
#define SA_CTA_R64 256      // 4 frames per CTA, one CTA per SM (255 registers): 64 / 128 / 256 threads = 418 / 426 / 435 Gsamples/s on C2
#endif

namespace sa {

struct R64Geo {
    static constexpr int N = 4096, P = 64, TPF = 64;
    static constexpr int CTA = SA_CTA_R64, FPC = CTA / TPF;
    static constexpr int SM_ELEMS = N + N / 64;              // one pad element per 64
    static constexpr int WROW = P + 2;
    static constexpr size_t EX_BYTES = (size_t)FPC * SM_ELEMS * sizeof(float2);
    static constexpr size_t WIN_BYTES = (size_t)TPF * WROW * sizeof(float);
    static constexpr size_t BAR_BYTES = (size_t)FPC * sizeof(uint64_t);
};

template <int DK, bool WIN>
__global__ void __launch_bounds__(R64Geo::CTA, 1)
spectrogram_r64_kernel(const SpecArgs a) {
    using G = R64Geo;
    using LD = Loader<float, DK>;
    using raw_t = typename LD::raw_t;
    constexpr int N = G::N, P = G::P, TPF = G::TPF, FPC = G::FPC;
    constexpr uint32_t FRAME_BYTES = N * sizeof(raw_t);
    static_assert(FRAME_BYTES <= G::SM_ELEMS * sizeof(float2), "raw frame must fit the exchange buffer");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int fl = threadIdx.x / TPF, t = threadIdx.x % TPF;
    float2* sm = reinterpret_cast<float2*>(smem_raw) + (size_t)fl * G::SM_ELEMS;
    const raw_t* raw = reinterpret_cast<const raw_t*>(sm);
    float* wsm = reinterpret_cast<float*>(smem_raw + G::EX_BYTES);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + G::EX_BYTES + (WIN ? G::WIN_BYTES : 0));
    const uint32_t bar = smem_u32(&bars[fl]);
    const uint32_t dst = smem_u32(sm);

    if constexpr (WIN) {        // window rows in first-stage pair order: factors of q and q + 32 adjacent
        const float* w = reinterpret_cast<const float*>(a.window);
        for (int i = threadIdx.x; i < N; i += G::CTA) {
            const int tt = i % TPF, e = i / TPF;             // sample tt + 64 e
            const int slot = e < P / 2 ? 2 * e : 2 * (e - P / 2) + 1;
            wsm[tt * G::WROW + slot] = __ldg(&w[i]);
        }
    }
    if (t == 0) mbar_init(bar, 1);
    __syncthreads();
    fence_proxy_async();
    const float* win = wsm + t * G::WROW;
    TwSeed<float> seed;
    {
        const float2* root = reinterpret_cast<const float2*>(a.aux);       // W_4096^j
        seed.om = __ldg(&root[t]);
        seed.oh = __ldg(&root[(32 * t) & (N - 1)]);
        seed.q_lo = __ldg(&root[(16 * t) & (N - 1)]);
        seed.q_hi = __ldg(&root[(48 * t) & (N - 1)]);
    }

    const long long n_blocks = (a.n_frames + FPC - 1) / FPC;
    const char* base = reinterpret_cast<const char*>(a.lp.base);
    auto frame_of = [&](long long fb) { return fb * FPC + fl; };
    auto readable_f = [&](long long frame) {
        return frame < a.n_frames && (a.start_sample + frame * a.hop + N <= a.n_samples);   // MainController.java:987
    };
    auto issue = [&](long long frame) {       // one thread of the frame
        mbar_expect_tx(bar, FRAME_BYTES);
        tma_load_1d(dst, base + (a.start_sample + frame * a.hop) * (long long)sizeof(raw_t), FRAME_BYTES, bar);
    };
    auto frame_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(fl + 1), "n"(TPF) : "memory"); };

    long long fb = blockIdx.x;
    if (fb < n_blocks && readable_f(frame_of(fb)) && t == 0) issue(frame_of(fb));
    uint32_t parity = 0;
    for (; fb < n_blocks; fb += gridDim.x) {
        const long long frame = frame_of(fb);
        const long long next = frame_of(fb + gridDim.x);
        const bool next_readable = (fb + gridDim.x < n_blocks) && readable_f(next);
        if (frame >= a.n_frames) continue;            // uniform over the frame's threads
        if (!readable_f(frame)) {                     // EOF row, no copy was issued for it
            store_fill<float, N>(a, frame, t);        // (Geo<float,4096>: 32 stores per thread cover the row twice over 64 threads)
            store_fill<float, N>(a, frame, t + TPF);
            if (next_readable && t == 0) issue(next);
            continue;
        }
        mbar_wait(bar, parity);
        parity ^= 1;
        float2 v[P];
        if (a.lp.swap) {
#pragma unroll
            for (int q = 0; q < P; q++) v[q] = LD::template decode<true>(a.lp, raw[t + TPF * q]);
        } else {
#pragma unroll
            for (int q = 0; q < P; q++) v[q] = LD::template decode<false>(a.lp, raw[t + TPF * q]);
        }
        // pass 0
        radix_fft<float, 64, 1, 0, P, WIN ? MUL_REAL : MUL_NONE, false>(v, win, nullptr, 0, seed);
        frame_sync();                                 // every thread has consumed the raw frame
        {
            float2* d = sm + 65 * t;                  // outputs 64 t + m, padded
#pragma unroll
            for (int m = 0; m < P; m++) d[m] = v[m];
        }
        frame_sync();
#pragma unroll
        for (int q = 0; q < P; q++) v[q] = sm[t + 65 * q];
        frame_sync();                                 // the exchange has been read back: the buffer is free
        if (next_readable && t == 0) {
            fence_proxy_async();
            issue(next);
        }
        // pass 1: twiddle W_N^(t m)
        radix_fft<float, 64, 1, 0, P, MUL_REC, false>(v, nullptr, nullptr, 0, seed);
        // epilogue: v[m] = X[t + 64 m]; shifted row index t + 64 m + 2048 (m < 32) or t + 64 (m - 32).  Two halves
        // of 32 bins keep the dB values of only one half live next to the spectrum (register budget).
        const size_t row = (size_t)frame * N;
#pragma unroll
        for (int h = 0; h < 2; h++) {
            float2 vh[P / 2];
#pragma unroll
            for (int m = 0; m < P / 2; m++) vh[m] = v[h * (P / 2) + m];
            float db[P / 2];
            if (a.db_mode == DBM_MAG_1E10) bins_to_db<float, P / 2, DBM_MAG_1E10>(vh, db);
            else bins_to_db<float, P / 2, DBM_POWER>(vh, db);
            const size_t off = row + t + (h == 0 ? N / 2 : 0);
            if (a.out_kind == OUT_F32_DB) {
                float* o = reinterpret_cast<float*>(a.out) + off;
#pragma unroll
                for (int m = 0; m < P / 2; m++) o[TPF * m] = db[m];
            } else if (a.out_kind == OUT_F64_DB) {
                double* o = reinterpret_cast<double*>(a.out) + off;
#pragma unroll
                for (int m = 0; m < P / 2; m++) o[TPF * m] = (double)db[m];
            } else {
                uint32_t* o = reinterpret_cast<uint32_t*>(a.out) + off;
                const float sc = a.inv_range, bi = a.cmap_bias;
                if (a.cmap == 1) {
#pragma unroll
                    for (int m = 0; m < P / 2; m++) o[TPF * m] = colormap_px<1>(db[m], sc, bi);
                } else {
#pragma unroll
                    for (int m = 0; m < P / 2; m++) o[TPF * m] = colormap_px<0>(db[m], sc, bi);
                }
            }
        }
    }
}

template <int DK, bool WIN>
SpecKernelInfo make_spec_r64_info() {
    using G = R64Geo;
    SpecKernelInfo k;
    k.fn = (const void*)&spectrogram_r64_kernel<DK, WIN>;
    k.fn_level = nullptr;                     // its store code is its own: level rows take the mid kernel
    k.prec = 1; k.n = G::N; k.dk = DK; k.win = WIN ? 1 : 0;
    k.cta = G::CTA; k.fpc = G::FPC; k.minb = 1;
    k.smem = G::EX_BYTES + (WIN ? G::WIN_BYTES : 0) + G::BAR_BYTES;
    k.p = 64; k.np = 2; k.tma = 4;
    k.radix[0] = 64; k.radix[1] = 64; k.radix[2] = 1; k.radix[3] = 1;
    return k;
}

}  // namespace sa
