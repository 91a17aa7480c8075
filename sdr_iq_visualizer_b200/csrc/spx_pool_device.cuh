// spx_pool_device.cuh -- per-element math of the pooled spectrogram (K8, spx_pool.cu), host and device.
//
// Kept apart from the kernels so that a CPU harness (tests/emul/pool_emul.cu) runs exactly these functions.
#pragma once
#include <math.h>
#include <stdint.h>

namespace spx {

// The power |X|^2 a float32 dB row value d = 20 log10(|X| + eps) encodes: (10^(d/20) - eps)^2, clipped at 0.
// NaN stays NaN (the comparison is false for it), so a NaN frame makes its mean cell NaN as it does in welch_acc.
__host__ __device__ inline float pool_db_to_power(float d, float eps) {
    float a = exp10f(d * 0.05f) - eps;
    a = a < 0.f ? 0.f : a;
    return a * a;
}

// pooled row of a global frame index, pooled column of a bin (fftshift order)
__host__ __device__ inline long long pool_row_of(long long frame, long long frames_per_row) { return frame / frames_per_row; }
__host__ __device__ inline int pool_col_of(int bin, int bins_per_col) { return bin / bins_per_col; }

// frames pooled into row g of a capture of n_frames_total frames: K, or fewer in the last row
__host__ __device__ inline long long pool_row_frames(long long g, long long frames_per_row, long long n_frames_total) {
    const long long end = (g + 1) * frames_per_row;
    return (end < n_frames_total ? end : n_frames_total) - g * frames_per_row;
}

// mean detector: the dB of the mean power of a cell of n_frames x bins_per_col values whose power sum is `sum`
__host__ __device__ inline float pool_mean_db(double sum, long long n_frames, int bins_per_col, float eps) {
    return (float)(20.0 * log10(sqrt(sum / ((double)n_frames * (double)bins_per_col)) + (double)eps));
}

// peak detector: the accumulator holds the largest float32 dB value itself (dB is monotonic in power)
__host__ __device__ inline float pool_max_db(double acc) { return (float)acc; }

// uint8 level of a float32 dB value by the waterfall rule (SURVEY.md 8(a) A7), evaluated in float64:
// clip(floor((db - vmin) * (256 / (vmax - vmin))), 0, 255), NaN -> 0, +inf -> 255, -inf -> 0
__host__ __device__ inline uint8_t pool_level(float db, float vmin, float vmax) {
    const double pre = ((double)db - (double)vmin) * (256.0 / ((double)vmax - (double)vmin));
    if (pre != pre) return 0;
    const double q = floor(pre);
    return q <= 0.0 ? (uint8_t)0 : (q >= 255.0 ? (uint8_t)255 : (uint8_t)q);
}

}  // namespace spx
