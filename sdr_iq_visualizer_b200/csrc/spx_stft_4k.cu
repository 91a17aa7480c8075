// N = 4096 instantiations of the fused STFT kernel (K1).
#include "spx_stft2_kernel.cuh"

namespace spx {
int launch_stft_4k(StftLaunch& L) {
    // K1v2 by default; K1 (TMA-staged input, register twiddle bases, int16 -> float on the ALU pipe) when frames are not
    // 128-byte aligned, and for variant 12, the reference the tests hold K1v2 to
    if (L.variant != 12 && stft2_ok(L)) return launch_stft2(L);
    return launch_stft_n<4096, TW_REG, 2, true, TUNE_I2FP>(L);
}
}  // namespace spx
