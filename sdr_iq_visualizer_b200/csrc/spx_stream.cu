// spx_stream.cu -- the reference's per-buffer stream path in float64 on the GPU.
//
// /root/reference/app/sdr/streamer.py:119-121 computes, once per rx buffer (4096 samples by default, ~244 buffers/s at
// 1 MS/s), fftshift(fft(samples)) and 20*log10(|X| + 1e-12) in float64.  Throughput is irrelevant at that rate, parity is
// not: a float32 FFT cannot hold deep nulls of a strong-tone frame to 1e-4 of the noise floor (the round-1 margin on the
// reference's own golden frames was 16 %).  So the drop-in `stream_frame` runs this float64 kernel: one CTA per buffer,
// in-place radix-2 in shared memory with exactly rounded float64 twiddles, hypot + log10 in float64 -- the result agrees
// with numpy to ~1e-12 dB.  The batched / overlapped STFT path (K1, K2) stays float32: that is where the bandwidth is.
// Power-of-two n in [2, 8192]; other lengths keep the float32 plan path (Bluestein, K2).
#include <math.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "spx_plan.h"

namespace spx {

template <bool C128>
__global__ void __launch_bounds__(512) stream_frame_f64_kernel(const void* __restrict__ in, int n, int log2n, const double2* __restrict__ tw,
                                                               double eps, double* __restrict__ power_db, double2* __restrict__ spec,
                                                               unsigned char* __restrict__ wf, double vmin, double q_scale) {
    extern __shared__ double2 buf[];
    // bit-reversed load (decimation in time)
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double2 x;
        if (C128) x = reinterpret_cast<const double2*>(in)[i];
        else {
            const float2 f = reinterpret_cast<const float2*>(in)[i];
            x = make_double2((double)f.x, (double)f.y);
        }
        buf[__brev((unsigned)i) >> (32 - log2n)] = x;
    }
    __syncthreads();
    for (int s = 1; s <= log2n; ++s) {
        const int half = 1 << (s - 1), tstep = n >> s;
        for (int i = threadIdx.x; i < n / 2; i += blockDim.x) {
            const int j = i & (half - 1), base = (i >> (s - 1)) << s;
            const double2 w = tw[j * tstep];        // exp(-2 pi i j / 2^s), rounded once from float64 cos / sin
            const double2 a = buf[base + j], b = buf[base + j + half];
            const double tr = __dsub_rn(__dmul_rn(b.x, w.x), __dmul_rn(b.y, w.y));
            const double ti = __dadd_rn(__dmul_rn(b.x, w.y), __dmul_rn(b.y, w.x));
            buf[base + j] = make_double2(a.x + tr, a.y + ti);
            buf[base + j + half] = make_double2(a.x - tr, a.y - ti);
        }
        __syncthreads();
    }
    // fftshift: output index j <- bin (j + n/2) mod n  (streamer.py:119); dB as streamer.py:121
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        const double2 X = buf[(j + n / 2) & (n - 1)];
        if (spec) spec[j] = X;
        const double db = 20.0 * log10(hypot(X.x, X.y) + eps);
        if (power_db) power_db[j] = db;
        if (wf) {
            const double q = floor((db - vmin) * q_scale);
            wf[j] = (unsigned char)(q != q ? 0.0 : fmin(fmax(q, 0.0), 255.0));
        }
    }
}

// the device table of n/2 float64 twiddles exp(-2 pi i k / n) of ctx's device
static int stream_twiddles(DeviceCtx* ctx, int n, double2** out) {
    auto it = ctx->tw64.find(n);
    if (it != ctx->tw64.end()) { *out = it->second; return SPX_OK; }
    std::vector<double2> h((size_t)(n / 2 > 0 ? n / 2 : 1));
    const double two_pi = 6.283185307179586476925286766559;
    for (int k = 0; k < n / 2; ++k) {
        // exact at the octants: cos / sin of k/n turns reduced to the first octant keeps every entry within 1 ulp
        const double a = -two_pi * (double)k / (double)n;
        h[k] = make_double2(cos(a), sin(a));
    }
    if (n >= 4) h[n / 4] = make_double2(0.0, -1.0);
    if (n >= 1) h[0] = make_double2(1.0, 0.0);
    double2* d = nullptr;
    SPX_CUDA(cudaMalloc(&d, h.size() * sizeof(double2)));
    SPX_CUDA(cudaMemcpy(d, h.data(), h.size() * sizeof(double2), cudaMemcpyHostToDevice));
    ctx->tw64[n] = d;
    *out = d;
    return SPX_OK;
}

}  // namespace spx

using namespace spx;

extern "C" int spx_stream_frame_f64(int device, int mem, const void* samples, int in_is_c128, int n, double eps, double* power_db_out,
                                    double* spec_out, uint8_t* wf_row, double vmin, double vmax, void* stream) {
    if (!samples || (!power_db_out && !spec_out && !wf_row)) return spx_set_error(SPX_E_INVALID, "NULL argument");
    if (n < 2 || n > 8192 || (n & (n - 1)) != 0) return spx_set_error(SPX_E_UNSUPPORTED, "spx_stream_frame_f64: n must be a power of two in [2, 8192], got %d", n);
    if (wf_row && !(vmax > vmin)) return spx_set_error(SPX_E_INVALID, "wf_row needs vmax > vmin");
    if (mem != SPX_MEM_HOST && mem != SPX_MEM_DEVICE) return spx_set_error(SPX_E_INVALID, "unknown mem %d", mem);
    DeviceCtx* ctx;
    SPX_TRY(device_ctx(device, &ctx));
    std::lock_guard<std::mutex> g(ctx->mu);
    double2* tw = nullptr;
    SPX_TRY(stream_twiddles(ctx, n, &tw));
    int log2n = 0;
    while ((1 << log2n) < n) ++log2n;
    cudaStream_t st = mem == SPX_MEM_HOST ? ctx->st : (cudaStream_t)stream;
    const size_t in_bytes = (size_t)n * (in_is_c128 ? 16 : 8);
    const void* d_in = samples;
    double* d_db = power_db_out;
    double2* d_spec = reinterpret_cast<double2*>(spec_out);
    unsigned char* d_wf = wf_row;
    if (mem == SPX_MEM_HOST) {
        void* part[4];
        SPX_TRY(ctx->carve({in_bytes, (size_t)n * sizeof(double), (size_t)n * sizeof(double2), (size_t)n}, part));
        SPX_CUDA(cudaMemcpyAsync(part[0], samples, in_bytes, cudaMemcpyHostToDevice, st));
        d_in = part[0];
        d_db = power_db_out ? (double*)part[1] : nullptr;
        d_spec = spec_out ? (double2*)part[2] : nullptr;
        d_wf = wf_row ? (unsigned char*)part[3] : nullptr;
    }
    const size_t smem = (size_t)n * sizeof(double2);
    auto kern = in_is_c128 ? stream_frame_f64_kernel<true> : stream_frame_f64_kernel<false>;
    SPX_TRY(kernel_setup((const void*)kern, 512, 8192 * sizeof(double2), nullptr));
    const double q_scale = wf_row ? 256.0 / (vmax - vmin) : 0.0;
    kern<<<1, n >= 1024 ? 512 : (n >= 64 ? n / 2 : 32), smem, st>>>(d_in, n, log2n, tw, eps, d_db, d_spec, d_wf, vmin, q_scale);
    SPX_CUDA(cudaGetLastError());
    if (mem == SPX_MEM_HOST) {
        if (power_db_out) SPX_CUDA(cudaMemcpyAsync(power_db_out, d_db, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
        if (spec_out) SPX_CUDA(cudaMemcpyAsync(spec_out, d_spec, (size_t)n * sizeof(double2), cudaMemcpyDeviceToHost, st));
        if (wf_row) SPX_CUDA(cudaMemcpyAsync(wf_row, d_wf, (size_t)n, cudaMemcpyDeviceToHost, st));
        SPX_CUDA(cudaStreamSynchronize(st));
    }
    return SPX_OK;
}
