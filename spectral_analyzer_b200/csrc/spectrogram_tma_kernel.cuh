// spectrogram_tma_kernel.cuh -- one-warp-per-frame spectrogram with TMA-staged frames.
//
// Same arithmetic and output as spectrogram_kernel (spectrogram_kernel.cuh) for the plans where a
// frame is owned by one warp (TPF == 32, i.e. the 1024-point FP32 plan), but the samples do not
// travel through LDG/L1: lane 0 of every warp issues ONE bulk asynchronous copy
// (cp.async.bulk global -> shared, completion on an mbarrier) that lands the warp's NEXT frame in
// the warp's own exchange buffer while pass 1 and the dB epilogue of the current frame run.  The
// raw frame and the Stockham exchange alias the same shared memory: the raw samples are consumed
// into registers before the exchange of that frame overwrites them, and the next copy is issued
// only after the exchange has been read back.
// Requires 16-byte aligned frame starts and sizes: the host takes this kernel when
// base, start_sample*bps and hop*bps are multiples of 16 and falls back to spectrogram_kernel.
#pragma once
#include "spectrogram_kernel.cuh"

#ifndef SA_TMA_EVICT_LAST
#define SA_TMA_EVICT_LAST 0
#endif
#ifndef SA_TMA_BLOCKS_PER_STEP
#define SA_TMA_BLOCKS_PER_STEP 1
#endif

namespace sa {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
#if SA_TMA_EVICT_LAST
    // overlapping frames read every sample twice: ask L2 to keep the lines until the second read
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
#else
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
#endif
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

#define SA_KERNEL_NAME spectrogram_tma_kernel
#define SA_KERNEL_LVL false
#include "spectrogram_tma_kernel_body.inc"
// level rows (OUT_LEVEL8, persistence spectra)
#define SA_KERNEL_NAME spectrogram_tma_level_kernel
#define SA_KERNEL_LVL true
#include "spectrogram_tma_kernel_body.inc"

template <typename T, int N, int DK, bool WIN>
SpecKernelInfo make_spec_tma_info(int prec) {
    SpecKernelInfo k = make_spec_info<T, N, DK, WIN>(prec);
    k.fn = (const void*)&spectrogram_tma_kernel<T, N, DK, WIN>;
    k.fn_level = (const void*)&spectrogram_tma_level_kernel<T, N, DK, WIN>;
    k.smem = Geo<T, N>::SMEM_BYTES + (WIN ? Geo<T, N>::WIN_BYTES : 0) + Geo<T, N>::FPC * sizeof(uint64_t);
    k.tma = 1;
    return k;
}

}  // namespace sa
