// CPU harness of the channelizer math (csrc/spx_chan_device.cuh): K10's fold, index maps and the STFT's FFT phases, run on
// the host so that tests/test_channelizer_cpu.py can hold them to tests/chan_ref.py and the GPU tests can compare K10 with
// them.
#include <vector>

#include "../../sdr_iq_visualizer_b200/csrc/spx_chan_device.cuh"
#include "../../sdr_iq_visualizer_b200/csrc/spx_tables.h"

template <int M>
static void run(const float2* xs, long long L, unsigned long long first, const float* g, int T, int D, int tb,
                float2* out, long long out_stride, float2* fold_out) {
    const long long n_out = (L - T) / D + 1;
    const std::vector<float2> tw = spx::build_twiddles(M);
    std::vector<float2> fold(M), y(M);
    for (long long m = 0; m < n_out; ++m) {
        const unsigned cls0 = spx::chan_cls0(first, m, D, M);
        for (int ft = 0; ft < M / 16; ++ft) {
            float2 v[16];
            for (int t = 0; t < 16; ++t) v[t] = make_float2(0.f, 0.f);
            // the whole input as the "ring": window offset j of output m is sample mD + j; the window in blocks of tb
            // offsets as the kernel's blocked mode folds it (tb = T: at once, as the ring mode does)
            for (int j_lo = 0; j_lo < T; j_lo += tb)
                spx::chan_fold<M>(v, ft, g, j_lo, T - j_lo < tb ? T : j_lo + tb, xs + m * D, 1 << 30, 0, cls0);
            for (int t = 0; t < 16; ++t) fold[ft + t * (M / 16)] = v[t];
        }
        if (fold_out)
            for (int r = 0; r < M; ++r) fold_out[m * M + r] = fold[r];
        spx::chan_fft_host<M>(fold.data(), tw.data(), y.data());
        for (int j = 0; j < M; ++j) out[j * out_stride + m] = y[j];
    }
}

extern "C" {

// x interleaved float32 (fmt 0) or int16 (fmt 1), taps h[0 .. T - 1] float32; out [M][out_stride] complex64;
// fold_out (optional) [n_out][M] the fold v_m[r] in natural class order; tb: window offsets per fold block (<= 0: T)
int emul_chan(const void* x, int fmt, float scale, long long L, unsigned long long first_sample, const float* h, int T,
              int M, int D, float* out, long long out_stride, float* fold_out, int tb) {
    if (L < T) return 0;
    std::vector<float2> xs((size_t)L);
    for (long long n = 0; n < L; ++n) {
        const float xr = fmt ? (float)((const short*)x)[2 * n] : ((const float*)x)[2 * n];
        const float xi = fmt ? (float)((const short*)x)[2 * n + 1] : ((const float*)x)[2 * n + 1];
        xs[(size_t)n] = make_float2(spx::ddc_mul(xr, scale), spx::ddc_mul(xi, scale));
    }
    std::vector<float> g((size_t)T);
    for (int j = 0; j < T; ++j) g[(size_t)j] = h[T - 1 - j];
    float2* o = (float2*)out;
    float2* fo = (float2*)fold_out;
    if (tb <= 0 || tb > T) tb = T;
    switch (M) {
        case 16: run<16>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        case 32: run<32>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        case 64: run<64>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        case 128: run<128>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        case 256: run<256>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        case 512: run<512>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        case 1024: run<1024>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        case 2048: run<2048>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        case 4096: run<4096>(xs.data(), L, first_sample, g.data(), T, D, tb, o, out_stride, fo); break;
        default: return -1;
    }
    return 0;
}

}
