// spx_bluestein.cu -- K5: STFT for frame lengths that are not a power of two (or shorter than 16).
//
// The reference transforms whatever `rx_buffer_size` the user configures with np.fft.fft
// (/root/reference/app/sdr/streamer.py:8-10,114-119; pocketfft handles any length).  The shared-memory Stockham
// kernels here are power-of-two only, so other lengths go through Bluestein's chirp-z identity on top of them:
//
//     X[k] = c[k] * sum_n (x[n] w[n] c[n]) * conj(c)[k - n],      c[n] = exp(-i pi n^2 / N)
//
// i.e. one circular convolution of length M = 2^ceil(log2(2N - 1)), evaluated with two M-point FFTs of the inner
// power-of-two plan (the inverse as conj(FFT(conj(.)))/M) and the precomputed spectrum B = FFT_M(conj(c), wrapped).
//   pre  : a[f][n] = x[f*hop + n] * (w[n]*scale*c[n]) for n < N, 0 for N <= n < M      (unpack + window + chirp fused)
//   FFT_M: A = FFT(a)                      (inner plan, complex rows out, fftshift order)
//   mul  : Y = conj(A * B)                 (B stored in the same fftshift order)
//   FFT_M: Z = FFT(Y)                      -> conv[n] = conj(Z[n]) / M
//   post : X[k] = c[k] * conv[k], k < N;  |X|^2 -> dB -> fftshift(N) -> rows / Welch / max-hold / u8 (fused epilogue)
// Chirp phases are reduced exactly in integers (n^2 mod 2N) and evaluated in float64 on the host; B is computed with a
// float64 FFT on the host at plan creation.
#include <math.h>
#include <string.h>

#include <vector>

#include "spx_plan.h"
#include "spx_stft_device.cuh"

namespace spx {

struct BluParams {
    const void* in;
    long long sample0;     // first sample of the first frame of this batch
    int hop, n, m, frames;
    const float2* wc;      // [N] window * scale * chirp
    const float2* chirp;   // [N] chirp / M (post-multiply, includes the 1/M of the inverse transform)
    const float2* bspec;   // [M] FFT_M(b) in fftshift order
    float2* buf_a;         // [frames][M]
    float2* buf_b;         // [frames][M]
    long long row0;
    float* db_rows;
    unsigned char* wf_rows;
    float2* spec_rows;
    double* welch_acc;
    float* maxhold;
    float db_eps, q_a, q_b;
    int sys_atomics;
    int frames_per_chunk;
};

template <int FMT>
__global__ void __launch_bounds__(256) blu_pre_kernel(const BluParams p) {
    const long long total = (long long)p.frames * p.m;
    for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const int f = (int)(i / p.m), n = (int)(i - (long long)f * p.m);
        float2 r = make_float2(0.f, 0.f);
        if (n < p.n) {
            const long long s = p.sample0 + (long long)f * p.hop + n;
            const float2 x = FMT == FMT_CF32 ? ld_stream_cf32(reinterpret_cast<const float2*>(p.in) + s)
                                             : ld_stream_ci16<TUNE_I2FP>(reinterpret_cast<const short2*>(p.in) + s);
            r = cmul(x, __ldg(p.wc + n));
        }
        p.buf_a[i] = r;
    }
}

__global__ void __launch_bounds__(256) blu_mul_kernel(const BluParams p) {
    const long long total = (long long)p.frames * p.m;
    for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
        const int j = (int)(i & (long long)(p.m - 1));
        const float2 y = cmul(p.buf_b[i], __ldg(p.bspec + j));
        // un-shift while writing: the second FFT must see natural bin order.  position j <-> bin (j + M/2) mod M
        const long long dst = (i - j) + ((j + p.m / 2) & (p.m - 1));
        p.buf_a[dst] = make_float2(y.x, -y.y);
    }
}

// one thread per output position jj (fftshift order of length N), looping over the frames of its chunk
template <bool ACC>
__global__ void __launch_bounds__(256) blu_post_kernel(const BluParams p) {
    const int jj = blockIdx.x * 256 + threadIdx.x;
    if (jj >= p.n) return;
    // np.fft.fftshift: out[jj] = X[(jj - N//2) mod N]
    int k = jj - p.n / 2;
    if (k < 0) k += p.n;
    const float2 c = __ldg(p.chirp + k);
    const int zpos = (k + p.m / 2) & (p.m - 1);   // Z is in fftshift order of length M
    const int f_lo = blockIdx.y * p.frames_per_chunk;
    const int f_hi = min(p.frames, f_lo + p.frames_per_chunk);
    float sum = 0.f, mx = 0.f;
    for (int f = f_lo; f < f_hi; ++f) {
        const float2 z = p.buf_b[(long long)f * p.m + zpos];
        const float2 X = cmul(make_float2(z.x, -z.y), c);
        const long long o = (p.row0 + f) * (long long)p.n + jj;
        if (p.spec_rows) p.spec_rows[o] = X;
        const float pw = X.x * X.x + X.y * X.y;
        if (ACC) { sum += pw; mx = fmaxf(mx, pw); }
        if (p.db_rows || p.wf_rows) {
            const float y = 2.0f * fast_log2(fast_sqrt(pw) + p.db_eps);   // log2 of the eps-corrected power
            if (p.db_rows) p.db_rows[o] = (0.5f * SPX_DB_PER_LOG2) * y;
            if (p.wf_rows) p.wf_rows[o] = (unsigned char)sat_floor_u8(quant_pre(y, p.q_a, p.q_b));
        }
    }
    if (ACC) flush_acc(p.welch_acc, p.maxhold, jj, sum, mx, p.sys_atomics);
}

// ------------------------------------------------------------------ host side
static void fft_f64(std::vector<double>& re, std::vector<double>& im) {   // iterative radix-2, plan creation only
    const size_t n = re.size();
    for (size_t i = 1, j = 0; i < n; ++i) {
        size_t bit = n >> 1;
        for (; j & bit; bit >>= 1) j ^= bit;
        j ^= bit;
        if (i < j) { std::swap(re[i], re[j]); std::swap(im[i], im[j]); }
    }
    const double two_pi = 6.283185307179586476925286766559;
    for (size_t len = 2; len <= n; len <<= 1) {
        const size_t half = len >> 1;
        std::vector<double> wr(half), wi(half);
        for (size_t k = 0; k < half; ++k) { wr[k] = cos(-two_pi * (double)k / (double)len); wi[k] = sin(-two_pi * (double)k / (double)len); }
        for (size_t i = 0; i < n; i += len)
            for (size_t k = 0; k < half; ++k) {
                const double ur = re[i + k], ui = im[i + k];
                const double vr = re[i + k + half] * wr[k] - im[i + k + half] * wi[k];
                const double vi = re[i + k + half] * wi[k] + im[i + k + half] * wr[k];
                re[i + k] = ur + vr; im[i + k] = ui + vi;
                re[i + k + half] = ur - vr; im[i + k + half] = ui - vi;
            }
    }
}

int bluestein_plan_init(spx_plan* pl) {
    const int n = pl->cfg.nfft;
    int m = 16;
    while (m < 2 * n - 1) m <<= 1;
    pl->blu_m = m;
    // inner power-of-two plan: rect window, cf32, hop = M, complex rows
    spx_plan_config ic = pl->cfg;
    ic.nfft = m; ic.hop = m; ic.window = SPX_WINDOW_RECT; ic.in_fmt = SPX_FMT_CF32; ic.in_scale = 1.0f; ic.variant = 0;
    SPX_TRY(spx_plan_create(&pl->blu_inner, &ic));
    const double pi = 3.14159265358979323846264338327950288;
    std::vector<double> cr((size_t)n), ci((size_t)n);
    for (int i = 0; i < n; ++i) {
        const long long q = ((long long)i * i) % (2ll * n);   // exact phase reduction
        const double a = -pi * (double)q / (double)n;
        cr[i] = cos(a); ci[i] = sin(a);
    }
    std::vector<float2> wc((size_t)n), ch((size_t)n);
    for (int i = 0; i < n; ++i) {
        const double w = pl->win64[i] * (double)pl->cfg.in_scale;
        wc[i] = make_float2((float)(w * cr[i]), (float)(w * ci[i]));
        ch[i] = make_float2((float)(cr[i] / (double)m), (float)(ci[i] / (double)m));
    }
    std::vector<double> br((size_t)m, 0.0), bi((size_t)m, 0.0);
    for (int i = 0; i < n; ++i) {
        br[i] = cr[i]; bi[i] = -ci[i];
        if (i) { br[(size_t)m - i] = cr[i]; bi[(size_t)m - i] = -ci[i]; }
    }
    fft_f64(br, bi);
    std::vector<float2> bs((size_t)m);
    for (int j = 0; j < m; ++j) {
        const int bin = (j + m / 2) & (m - 1);
        bs[j] = make_float2((float)br[bin], (float)bi[bin]);
    }
    SPX_CUDA(cudaMalloc(&pl->d_blu, (size_t)(2 * n + m) * sizeof(float2)));
    SPX_CUDA(cudaMemcpy(pl->d_blu, wc.data(), (size_t)n * sizeof(float2), cudaMemcpyHostToDevice));
    SPX_CUDA(cudaMemcpy(pl->d_blu + n, ch.data(), (size_t)n * sizeof(float2), cudaMemcpyHostToDevice));
    SPX_CUDA(cudaMemcpy(pl->d_blu + 2 * n, bs.data(), (size_t)m * sizeof(float2), cudaMemcpyHostToDevice));
    return SPX_OK;
}

int bluestein_launch_stream(spx_plan* pl, const void* in, long long frames, long long row0, const StftOut& out,
                            cudaStream_t st) {
    const int n = pl->cfg.nfft, m = pl->blu_m;
    const size_t frame_bytes = (size_t)m * sizeof(float2);
    long long fb = (long long)((128u << 20) / frame_bytes);
    if (fb < 1) fb = 1;
    if (fb > frames) fb = frames;
    SPX_TRY(pl->st_big.reserve((size_t)(2 * fb) * frame_bytes));
    BluParams p;
    memset(&p, 0, sizeof(p));
    p.in = in;
    p.hop = pl->cfg.hop;
    p.n = n;
    p.m = m;
    p.wc = pl->d_blu;
    p.chirp = pl->d_blu + n;
    p.bspec = pl->d_blu + 2 * n;
    p.buf_a = (float2*)pl->st_big.ptr;
    p.buf_b = p.buf_a + (size_t)fb * m;
    p.db_rows = out.db;
    p.wf_rows = out.wf;
    p.spec_rows = out.spec;
    p.welch_acc = out.welch;
    p.maxhold = out.maxhold;
    p.db_eps = pl->cfg.db_eps;
    p.q_a = out.q_a();
    p.q_b = out.q_b();
    p.sys_atomics = out.sys_atomics;
    const bool acc = out.welch != nullptr || out.maxhold != nullptr;
    const int sms = pl->sm_count;
    StftOut inner;   // the inner power-of-two transform: spectrum rows in buf_b
    inner.spec = p.buf_b;
    for (long long f0 = 0; f0 < frames; f0 += fb) {
        p.frames = (int)(frames - f0 < fb ? frames - f0 : fb);
        p.sample0 = f0 * pl->cfg.hop;
        p.row0 = row0 + f0;
        const long long total = (long long)p.frames * m;
        const unsigned g1 = (unsigned)((total + 255) / 256 < (long long)sms * 16 ? (total + 255) / 256 : (long long)sms * 16);
        if (pl->cfg.in_fmt == SPX_FMT_CF32) blu_pre_kernel<FMT_CF32><<<g1, 256, 0, st>>>(p);
        else blu_pre_kernel<FMT_CI16><<<g1, 256, 0, st>>>(p);
        SPX_CUDA(cudaGetLastError());
        SPX_TRY(stft_launch_device(pl->blu_inner, p.buf_a, 1, 0, p.frames, inner, st));
        blu_mul_kernel<<<g1, 256, 0, st>>>(p);
        SPX_CUDA(cudaGetLastError());
        SPX_TRY(stft_launch_device(pl->blu_inner, p.buf_a, 1, 0, p.frames, inner, st));
        const int bx = (n + 255) / 256;
        int chunks = (sms * 8 + bx - 1) / bx;
        if (chunks > p.frames) chunks = p.frames;
        if (chunks < 1) chunks = 1;
        p.frames_per_chunk = (p.frames + chunks - 1) / chunks;
        const dim3 g3((unsigned)bx, (unsigned)((p.frames + p.frames_per_chunk - 1) / p.frames_per_chunk));
        if (acc) blu_post_kernel<true><<<g3, 256, 0, st>>>(p);
        else blu_post_kernel<false><<<g3, 256, 0, st>>>(p);
        SPX_CUDA(cudaGetLastError());
    }
    return SPX_OK;
}

}  // namespace spx
