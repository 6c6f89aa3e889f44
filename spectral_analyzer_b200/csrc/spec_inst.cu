// spec_inst.cu -- explicit instantiations of spectrogram_kernel, one object file per
// (precision, nfft) so the build parallelises: compiled with -DSA_INST_PREC=1|2 -DSA_INST_N=<nfft>.
#include "spectrogram_tma_kernel.cuh"
#include "spectrogram_mid_kernel.cuh"
#include "spectrogram_r64_kernel.cuh"

#ifndef SA_INST_PREC
#error "compile with -DSA_INST_PREC=1|2 -DSA_INST_N=<nfft>"
#endif

namespace sa {
namespace {
struct Registrar {
    Registrar() {
#if SA_INST_PREC == 1
        // FP32 arithmetic: cf32 / ci16 / cu8+ci8 inputs, with and without a window multiply
        register_spec_kernel(make_spec_info<float, SA_INST_N, DK_CF32, false>(1));
        register_spec_kernel(make_spec_info<float, SA_INST_N, DK_CF32, true>(1));
        register_spec_kernel(make_spec_info<float, SA_INST_N, DK_CI16, false>(1));
        register_spec_kernel(make_spec_info<float, SA_INST_N, DK_CI16, true>(1));
        register_spec_kernel(make_spec_info<float, SA_INST_N, DK_C8, false>(1));
        register_spec_kernel(make_spec_info<float, SA_INST_N, DK_C8, true>(1));
#if SA_INST_N == 1024
        // one warp per frame: TMA-staged variants, taken when the frames are 16-byte aligned
        register_spec_kernel(make_spec_tma_info<float, SA_INST_N, DK_CF32, false>(1));
        register_spec_kernel(make_spec_tma_info<float, SA_INST_N, DK_CF32, true>(1));
        register_spec_kernel(make_spec_tma_info<float, SA_INST_N, DK_CI16, false>(1));
        register_spec_kernel(make_spec_tma_info<float, SA_INST_N, DK_CI16, true>(1));
        register_spec_kernel(make_spec_tma_info<float, SA_INST_N, DK_C8, false>(1));
        register_spec_kernel(make_spec_tma_info<float, SA_INST_N, DK_C8, true>(1));
#endif
#if SA_INST_N == 8192
        // small-radix-first plan with 128-bit loads, taken when the frames are 16-byte aligned (at 8192 points without
        // the next-frame staging below: it measured up to 19 % slower there)
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_CF32, false, false>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_CF32, true, false>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_CI16, false, false>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_CI16, true, false>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_C8, false, false>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_C8, true, false>());
#elif SA_INST_N >= 2048
        // small-radix-first plan with 128-bit loads and the next frame staged asynchronously (cp.async) under pass 2 and
        // the epilogue, taken when the frames are 16-byte aligned
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_CF32, false, true>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_CF32, true, true>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_CI16, false, true>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_CI16, true, true>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_C8, false, true>());
        register_spec_kernel(make_spec_mid_info<SA_INST_N, DK_C8, true, true>());
#endif
#if SA_INST_N == 4096
        // two-pass radix-64 plan (default for cf32 / ci16 input with 16-byte aligned frames)
        register_spec_kernel(make_spec_r64_info<DK_CF32, false>());
        register_spec_kernel(make_spec_r64_info<DK_CF32, true>());
        register_spec_kernel(make_spec_r64_info<DK_CI16, false>());
        register_spec_kernel(make_spec_r64_info<DK_CI16, true>());
#endif
#else
        // FP64 arithmetic (cf64 input, or any input when the caller asks for SA_PREC_F64);
        // always windowed -- a rectangular window is a table of ones
        register_spec_kernel(make_spec_info<double, SA_INST_N, DK_CF32, true>(2));
        register_spec_kernel(make_spec_info<double, SA_INST_N, DK_CI16, true>(2));
        register_spec_kernel(make_spec_info<double, SA_INST_N, DK_C8, true>(2));
        register_spec_kernel(make_spec_info<double, SA_INST_N, DK_CF64, true>(2));
#endif
    }
};
static Registrar registrar_instance;
}  // namespace
}  // namespace sa
