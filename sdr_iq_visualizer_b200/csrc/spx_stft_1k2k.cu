// N = 1024, 2048 instantiations of the fused STFT kernel (K1).
#include "spx_stft2_kernel.cuh"

namespace spx {
int launch_stft_1k2k(StftLaunch& L) {
    if (L.variant != 12 && stft2_ok(L)) return launch_stft2(L);   // K1v2 (default); variant 12 = K1, the tests' reference for K1v2
    // measured on B200 (tools/sweep_1k2k.py): N = 1024 rows-only shapes gain 5 % from the shared-memory table
    // (404 -> 424 GS/s, 78 % of HBM); with accumulators, and for N = 2048 (16 KB table), the L1 path is faster
    const bool acc = L.p.welch_acc != nullptr || L.p.maxhold != nullptr;
    if (L.nfft == 1024 && !acc) return launch_stft_n<1024, TW_SMEM, 2, true, TUNE_I2FP>(L);
    switch (L.nfft) {
        case 1024: return launch_stft_n<1024, TW_LDG, 2, true, TUNE_I2FP>(L);
        case 2048: return launch_stft_n<2048, TW_LDG, 2, true, TUNE_I2FP>(L);
        default: return spx_set_error(SPX_E_UNSUPPORTED, "nfft %d", L.nfft);
    }
}
}  // namespace spx
