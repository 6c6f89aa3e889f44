// spectrogram_mid_kernel.cuh -- FP32 spectrogram for nfft 2048 .. 16384 with 16-byte aligned frames.
//
// Same arithmetic contract and output as spectrogram_kernel (SpectralService.java:33-85 inside the frame
// loop of MainController.java:980-999), but the plan puts the SMALL radix first:
//   N = R0 * 32 * 32, R0 = N/1024 in {2, 4, 8, 16}, 32 points per thread, TPF = N/32 threads per frame.
//   pass 0  radix R0, S = 32/R0 butterflies per thread, window folded into the first stage.  Thread t owns
//           the S CONSECUTIVE samples S*t .. S*t+S-1 of each of the R0 slices of the frame, so the raw bytes
//           arrive as 128-bit loads (cu8: 8 samples per load) and the thread's 32 outputs are one
//           contiguous 256-byte block of the exchange buffer.
//   pass 1  radix 32; twiddles W_{32 R0}^{(t mod R0) m} come from a tiny shared-memory table (R0 x 32).
//   pass 2  radix 32; twiddles W_N^{t m} by the packed register recurrence seeded with W_N^t.
// Against the general plan (32 * 32 * R0: twiddle pairs for two passes from global memory) this removes
// every per-frame twiddle LDG and the scalar radix-R0 tail with its 8 distinct twiddle sets per thread.
// Exchange buffer: one pad element per 32 (physical index i + i/32) keeps all three access patterns at the
// two-wavefront minimum of 64-bit accesses (a warp moves 256 bytes; bank of an 8-byte element = physical index
// mod 16, so a pattern is conflict-free when the 32 lanes cover every residue exactly twice):
//   pass-0 write   lane t, fixed (i, m): logical 32 t + c  -> physical 33 t + c        : residues t + c      (each twice)
//   read-back      lane t, fixed q     : logical t + TPF q -> physical t + t/32 + const : consecutive         (each twice)
//   pass-1 write   lane t, fixed m     : logical (t/R0) 32 R0 + (t mod R0) + m R0
//                                        -> physical (t/R0) 33 R0 + (t mod R0) + const  : residues R0 (t/R0) + (t mod R0) = t
// (33 R0 = R0 mod 16 for every R0 in {2, 4, 8, 16}); the pass-2 input is the same read-back pattern.
#pragma once
#include "spectrogram_kernel.cuh"

#ifndef SA_CTA_MID
#define SA_CTA_MID 512
#endif
#ifndef SA_CTA_MID_4096
#define SA_CTA_MID_4096 512
#endif

namespace sa {

// Pass-1 twiddle recurrence from this transform length up.  8192 / 16384 gain 2 % (0.83 -> 0.81, 0.80 -> 0.79 ms); at 2048 the
// kernel is bound by the FP32 pipe, not by shared memory, and loses (cu8 2048 -> f32 dB 1.96 -> 2.23 ms, -> RGBA 4.57 -> 4.80 ms).
#ifndef SA_MID_REC1_MIN_N
#define SA_MID_REC1_MIN_N 8192
#endif
template <int N> struct MidGeo {
    static constexpr int P = 32, R0 = N / 1024, S = P / R0, TPF = N / P;
    // FPC consecutive frames per CTA step (16 warps; measured per size: 2048 -> 512 threads (C4 4.85 -> 4.76 ms); 4096 -> 512 threads together with the
    // staged variant (C2 417 -> 420, 50 % overlap 189 -> 210 Gsamples/s; without staging 128 threads were best))
    static constexpr int CTA = (N == 4096) ? SA_CTA_MID_4096 : (TPF > SA_CTA_MID ? TPF : SA_CTA_MID);
    static constexpr int FPC = CTA / TPF;
    static constexpr int MINB = 512 / CTA;
    static constexpr int SM_ELEMS = N + N / 32;
    static constexpr int WROW = P + 2;
    static constexpr size_t EX_BYTES = (size_t)FPC * SM_ELEMS * sizeof(float2);
    static constexpr size_t T1_BYTES = (size_t)16 * R0 * sizeof(float4);
    static constexpr size_t WIN_BYTES = (size_t)TPF * WROW * sizeof(float);
};

__device__ __forceinline__ int mid_pad(int i) { return i + (i >> 5); }

// barrier over the TPF threads of one frame (named barrier when a CTA holds several frames)
template <int TPF, int FPC> __device__ __forceinline__ void mid_sync(const int fl) {
    if constexpr (FPC == 1) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(fl + 1), "n"(TPF) : "memory");
}

__device__ __forceinline__ uint4 ldg_stream16(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg_stream8(const void* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ uint32_t ldg_stream4(const void* p) {
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

// decode of S consecutive samples held as raw words -> v[OFF + i], i < S (decode.cuh, same values bit for bit)
template <int DK, int S, bool SWAP, int OFF>
__device__ __forceinline__ void mid_decode_words(const LoadParams& lp, const uint32_t (&w)[S * bytes_per_iq_kind<DK>() / 4],
                                                 float2 (&v)[32]) {
#pragma unroll
    for (int i = 0; i < S; i++) {
        if constexpr (DK == DK_CF32) {
            v[OFF + i] = Loader<float, DK_CF32>::template decode<SWAP>(lp, make_uint2(w[2 * i], w[2 * i + 1]));
        } else if constexpr (DK == DK_CI16) {
            v[OFF + i] = Loader<float, DK_CI16>::template decode<SWAP>(lp, w[i]);
        } else {
            // two cu8/ci8 IQ pairs per word: byte -> bits 8..15 of a 2^23-exponent float (value 2^23 + 256 u),
            // then one exact FMA: (2^23 + 256 u) * 2^-15 - (256 + off) = u/128 - off   (off = 255/256 or 1)
            const uint32_t x = w[i / 2] ^ lp.c8_flip;
            const uint32_t sel = (i & 1) ? 0x7424u : 0x7404u;
            const float a = __uint_as_float(__byte_perm(x, 0x4B000000u, sel));
            const float b = __uint_as_float(__byte_perm(x, 0x4B000000u, sel + 0x10u));
            v[OFF + i] = make_float2(__fmaf_rn(a, 1.0f / 32768.0f, -lp.c8_c), __fmaf_rn(b, 1.0f / 32768.0f, -lp.c8_c));
        }
    }
}

// S consecutive samples starting at p (global memory, streaming loads) -> v[OFF + i]
template <int DK, int S, bool SWAP, int OFF>
__device__ __forceinline__ void mid_load_slice(const LoadParams& lp, const char* __restrict__ p, float2 (&v)[32]) {
    constexpr int BYTES = S * bytes_per_iq_kind<DK>();
    static_assert(BYTES >= 4 && BYTES % 4 == 0, "slice must be whole words");
    uint32_t w[BYTES / 4];
    if constexpr (BYTES >= 16) {
#pragma unroll
        for (int i = 0; i < BYTES / 16; i++) {
            const uint4 x = ldg_stream16(p + 16 * i);
            w[4 * i] = x.x; w[4 * i + 1] = x.y; w[4 * i + 2] = x.z; w[4 * i + 3] = x.w;
        }
    } else if constexpr (BYTES == 8) {
        const uint2 x = ldg_stream8(p);
        w[0] = x.x; w[1] = x.y;
    } else {
        w[0] = ldg_stream4(p);
    }
    mid_decode_words<DK, S, SWAP, OFF>(lp, w, v);
}

template <int DK, int N, bool SWAP, int M = 0>
__device__ __forceinline__ void mid_load_frame(const LoadParams& lp, const char* __restrict__ frame_base, const int t,
                                               float2 (&v)[32]) {
    using G = MidGeo<N>;
    constexpr int bps = bytes_per_iq_kind<DK>();
    mid_load_slice<DK, G::S, SWAP, G::S * M>(lp, frame_base + ((size_t)M * (N / G::R0) + (size_t)G::S * t) * bps, v);
    if constexpr (M + 1 < G::R0) mid_load_frame<DK, N, SWAP, M + 1>(lp, frame_base, t, v);
}

// ---- asynchronous staging of the NEXT frame (cp.async, one 16/8/4-byte chunk per thread and step) ----
// Chunk c = m*CH + i of thread t lands at byte ((c*TPF) + t)*CHB of the frame's exchange buffer: consecutive threads,
// consecutive chunks -> conflict-free both for the asynchronous writes and for the 128-bit reads of the same
// thread one frame later (a thread only ever reads back what it staged itself: no barrier on that side).
template <int DK, int N> struct MidStage {
    using G = MidGeo<N>;
    static constexpr int bps = bytes_per_iq_kind<DK>();
    static constexpr int BYTES = G::S * bps;                 // bytes of one slice per thread
    static constexpr int CHB = BYTES >= 16 ? 16 : BYTES;     // chunk bytes
    static constexpr int CH = BYTES / CHB;                   // chunks per slice
    static_assert((size_t)N * bps <= (size_t)G::SM_ELEMS * sizeof(float2), "raw frame fits the exchange buffer");
};

template <int CHB> __device__ __forceinline__ void cp_async_chunk(uint32_t dst, const void* src) {
    if constexpr (CHB == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
    else if constexpr (CHB == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}

template <int DK, int N>
__device__ __forceinline__ void mid_stage_frame(const char* __restrict__ frame_base, const int t, const uint32_t sm_addr) {
    using G = MidGeo<N>;
    using ST = MidStage<DK, N>;
#pragma unroll
    for (int m = 0; m < G::R0; m++)
#pragma unroll
        for (int i = 0; i < ST::CH; i++)
            cp_async_chunk<ST::CHB>(sm_addr + (uint32_t)(((m * ST::CH + i) * G::TPF + t) * ST::CHB),
                                    frame_base + ((size_t)m * (N / G::R0) + (size_t)G::S * t) * ST::bps + i * ST::CHB);
    asm volatile("cp.async.commit_group;" ::: "memory");
}

template <int DK, int N, bool SWAP, int M = 0>
__device__ __forceinline__ void mid_decode_staged(const LoadParams& lp, const unsigned char* __restrict__ stage, const int t,
                                                  float2 (&v)[32]) {
    using G = MidGeo<N>;
    using ST = MidStage<DK, N>;
    uint32_t w[ST::BYTES / 4];
#pragma unroll
    for (int i = 0; i < ST::CH; i++) {
        const unsigned char* p = stage + (size_t)((M * ST::CH + i) * G::TPF + t) * ST::CHB;
        if constexpr (ST::CHB == 16) {
            const uint4 x = *reinterpret_cast<const uint4*>(p);
            w[4 * i] = x.x; w[4 * i + 1] = x.y; w[4 * i + 2] = x.z; w[4 * i + 3] = x.w;
        } else if constexpr (ST::CHB == 8) {
            const uint2 x = *reinterpret_cast<const uint2*>(p);
            w[0] = x.x; w[1] = x.y;
        } else {
            w[0] = *reinterpret_cast<const uint32_t*>(p);
        }
    }
    mid_decode_words<DK, G::S, SWAP, G::S * M>(lp, w, v);
    if constexpr (M + 1 < G::R0) mid_decode_staged<DK, N, SWAP, M + 1>(lp, stage, t, v);
}

// The three passes of the small-radix-first plan on the registers of one frame.  In: v[i + S*m] = sample
// m*(N/R0) + S*t + i (already decoded); out: v[q] = X[t + TPF*q].  `sm` is the frame's exchange buffer, `win` the
// thread's window row (pair order), `t1_row` = pass-1 twiddle pairs + (t mod R0), seed = (W_N^t, W_N^(16 t)).
// REC1: the pass-1 twiddles W_{32 R0}^{(t mod R0) m} come from a packed register recurrence seeded by `seed1`
// (om = the m = 1 entry of the thread's table column, oh = om^16) instead of 16 LDS.128 per frame -- for callers bound by
// the shared-memory pipe (the Welch kernel: LSU wavefronts 68 %, FMA pipe 47 %).
template <int N, bool WIN, bool REC1 = false>
__device__ __forceinline__ void mid_fft_front(float2 (&v)[32], const int t, const int fl, float2* __restrict__ sm,
                                              const float* __restrict__ win, const TwPair<float>* __restrict__ t1_row,
                                              const TwSeed<float>& seed, const TwSeed<float>* seed1 = nullptr) {
    using G = MidGeo<N>;
    constexpr int P = 32, R0 = G::R0, S = G::S, TPF = G::TPF, FPC = G::FPC;
    // pass 0: S radix-R0 butterflies on v[i + S*m]
    RadixAll<float, R0, S, P, WIN ? MUL_REAL : MUL_NONE, false, 0>::run(v, win, nullptr, 0, seed);
    mid_sync<TPF, FPC>(fl);                  // the previous frame's exchange has been read back
    {
        float2* dst = sm + 33 * t;           // outputs j*R0 + m, j = S*t + i: the block [32 t, 32 t + 32)
#pragma unroll
        for (int i = 0; i < S; i++)
#pragma unroll
            for (int m = 0; m < R0; m++) dst[i * R0 + m] = v[i + S * m];
    }
    mid_sync<TPF, FPC>(fl);
#pragma unroll
    for (int q = 0; q < P; q++) v[q] = sm[mid_pad(t) + q * (TPF + TPF / 32)];

    // pass 1: radix 32, Ns = R0
    if constexpr (REC1) radix_fft<float, 32, 1, 0, P, MUL_REC, false>(v, nullptr, nullptr, 0, *seed1);
    else radix_fft<float, 32, 1, 0, P, MUL_CPX, true>(v, nullptr, t1_row, R0, seed);
    mid_sync<TPF, FPC>(fl);
    {
        float2* dst = sm + (t / R0) * (33 * R0) + (t % R0);
#pragma unroll
        for (int m = 0; m < 32; m++) dst[m * R0 + ((m * R0) >> 5)] = v[m];
    }
    mid_sync<TPF, FPC>(fl);
#pragma unroll
    for (int q = 0; q < P; q++) v[q] = sm[mid_pad(t) + q * (TPF + TPF / 32)];
}

// pass 2 (no shared memory): radix 32, Ns = 32 R0 = TPF, twiddle W_N^(t m) by recurrence
__device__ __forceinline__ void mid_fft_back(float2 (&v)[32], const TwSeed<float>& seed) {
    radix_fft<float, 32, 1, 0, 32, MUL_REC, false>(v, nullptr, nullptr, 0, seed);
}

template <int N, bool WIN, bool REC1 = false>
__device__ __forceinline__ void mid_fft(float2 (&v)[32], const int t, const int fl, float2* __restrict__ sm,
                                        const float* __restrict__ win, const TwPair<float>* __restrict__ t1_row,
                                        const TwSeed<float>& seed, const TwSeed<float>* seed1 = nullptr) {
    mid_fft_front<N, WIN, REC1>(v, t, fl, sm, win, t1_row, seed, seed1);
    mid_fft_back(v, seed);
}

// Copies the pass-1 twiddle pairs and (WIN) the window rows in first-stage pair order into shared memory;
// the caller synchronises the CTA afterwards.
template <int N, bool WIN>
__device__ __forceinline__ void mid_setup_tables(const void* __restrict__ t1_global, const void* __restrict__ window,
                                                 TwPair<float>* __restrict__ t1, float* __restrict__ wsm) {
    using G = MidGeo<N>;
    constexpr int P = 32, R0 = G::R0, S = G::S;
    const float4* src = reinterpret_cast<const float4*>(t1_global);
    float4* dst = reinterpret_cast<float4*>(t1);
    // (blockDim.x, not G::CTA: the Welch kernel also runs this plan with one segment per CTA; unroll 1 keeps the
    // compiler from computing a trip count by integer division)
#pragma unroll 1
    for (int i = threadIdx.x; i < 16 * R0; i += blockDim.x) dst[i] = __ldg(&src[i]);
    if constexpr (WIN) {
        const float* w = reinterpret_cast<const float*>(window);
#pragma unroll 1
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            // sample i = m*(N/R0) + S*tt + ii  ->  register e = ii + S*m of thread tt
            const int m = i / (N / R0), rem = i % (N / R0), tt = rem / S, ii = rem % S;
            const int e = ii + S * m;
            const int slot = e < P / 2 ? 2 * e : 2 * (e - P / 2) + 1;
            wsm[tt * G::WROW + slot] = __ldg(&w[i]);
        }
    }
}

// PF: the raw bytes of a slot's NEXT frame are staged asynchronously into the (then idle) exchange buffer while
// pass 2 and the epilogue of the current frame run, so no global-load latency sits on the per-frame critical
// path (it matters most where one or two frames occupy a whole SM: nfft 8192 / 16384).
#define SA_KERNEL_NAME spectrogram_mid_kernel
#define SA_KERNEL_LVL false
#include "spectrogram_mid_kernel_body.inc"
// level rows (OUT_LEVEL8, persistence spectra)
#define SA_KERNEL_NAME spectrogram_mid_level_kernel
#define SA_KERNEL_LVL true
#include "spectrogram_mid_kernel_body.inc"

template <int N, int DK, bool WIN, bool PF>
SpecKernelInfo make_spec_mid_info() {
    using G = MidGeo<N>;
    SpecKernelInfo k;
    k.fn = (const void*)&spectrogram_mid_kernel<N, DK, WIN, PF>;
    k.fn_level = (const void*)&spectrogram_mid_level_kernel<N, DK, WIN, PF>;
    k.prec = 1; k.n = N; k.dk = DK; k.win = WIN ? 1 : 0;
    k.cta = G::CTA; k.fpc = G::FPC; k.minb = G::MINB;
    k.smem = G::EX_BYTES + G::T1_BYTES + (WIN ? G::WIN_BYTES : 0);
#ifdef SA_MID_SMEM_PAD          // occupancy ablation: pad the request so that fewer CTAs fit an SM
    if (k.smem < (size_t)SA_MID_SMEM_PAD) k.smem = (size_t)SA_MID_SMEM_PAD;
#endif
    k.p = 32; k.np = 3; k.tma = PF ? 3 : 2;
    k.radix[0] = G::R0; k.radix[1] = 32; k.radix[2] = 32; k.radix[3] = 1;
    return k;
}

}  // namespace sa
