// spx_features.cu -- K3: the classifier's spectrum measurements on the GPU.
//
// Replaces the numpy feature extraction of /root/reference/app/processing/classifier.py:45-58
// (helpers :163-219): 20th-percentile noise floor (exact order statistics + numpy's lerp), peak /
// SNR, occupied-bandwidth edges at 3/10/20 dB (>=) and the simple classifier's strict 20 dB edges,
// spectral flatness, kurtosis, and the greedy min-distance peak pick (:200-212, a pure-Python loop
// in the reference).  One CTA of 1024 threads per spectrum; everything is evaluated in float64 with
// explicitly rounded operations so that thresholds compare exactly as numpy's do.
// The label rules and temporal smoothing (:60-161) stay on the host (scalar logic).
#include <float.h>
#include <math.h>
#include <string.h>

#include <mutex>

#include "spx_internal.h"
#include "spx_plan.h"

namespace spx {

constexpr int FT = 1024;  // threads per CTA

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide reductions through shared memory; every thread gets the result
__device__ double block_sum(double v, double* sh) {
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    double r = (threadIdx.x < FT / 32) ? sh[threadIdx.x] : 0.0;
    if (w == 0) r = warp_sum(r);
    if (threadIdx.x == 0) sh[0] = r;
    __syncthreads();
    return sh[0];
}
__device__ long long block_min_ll(long long v, long long* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { long long t = __shfl_xor_sync(0xffffffffu, v, o); v = t < v ? t : v; }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    long long r = (threadIdx.x < FT / 32) ? sh[threadIdx.x] : LLONG_MAX;
    if (w == 0) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { long long t = __shfl_xor_sync(0xffffffffu, r, o); r = t < r ? t : r; }
    }
    if (threadIdx.x == 0) sh[0] = r;
    __syncthreads();
    return sh[0];
}
__device__ long long block_max_ll(long long v, long long* sh) { return -block_min_ll(-v, sh); }

__device__ unsigned long long block_max_u64(unsigned long long v, unsigned long long* sh) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { unsigned long long t = __shfl_xor_sync(0xffffffffu, v, o); v = t > v ? t : v; }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) sh[w] = v;
    __syncthreads();
    unsigned long long r = sh[l];   // FT / 32 == 32 partials: every warp reduces them redundantly, no third barrier
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { unsigned long long t = __shfl_xor_sync(0xffffffffu, r, o); r = t > r ? t : r; }
    return r;
}
// three sums at once (every thread gets the results)
__device__ void block_sum3(double* v, double (*sh)[FT / 32]) {
#pragma unroll
    for (int q = 0; q < 3; ++q) v[q] = warp_sum(v[q]);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) { sh[0][w] = v[0]; sh[1][w] = v[1]; sh[2][w] = v[2]; }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 3; ++q) v[q] = warp_sum(sh[q][l]);
}
// eight integer minima at once
__device__ void block_min8(int* v, int (*sh)[FT / 32]) {
#pragma unroll
    for (int q = 0; q < 8; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[q] = min(v[q], __shfl_xor_sync(0xffffffffu, v[q], o));
    }
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    __syncthreads();
    if (l == 0) {
#pragma unroll
        for (int q = 0; q < 8; ++q) sh[q][w] = v[q];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        int r = sh[q][l];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r = min(r, __shfl_xor_sync(0xffffffffu, r, o));
        v[q] = r;
    }
}

// order-preserving map double -> uint64; every NaN, whatever its sign bit or payload, maps to the largest key, so NaN
// sorts last as in np.sort
__device__ __forceinline__ unsigned long long key_of(double x) {
    if (x != x) return ~0ull;
    unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double val_of(unsigned long long k) {
    unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

template <typename T>
__global__ void __launch_bounds__(FT, 1)
features_kernel(const T* __restrict__ data, int n, long long stride, spx_features* __restrict__ out,
                int* __restrict__ peaks, int peaks_cap, const spx_feature_opts opts) {
    __shared__ double shd[FT / 32];
    __shared__ double shd3[3][FT / 32];
    __shared__ long long shl[FT / 32];
    __shared__ unsigned long long shu[FT / 32];
    __shared__ int shi8[8][FT / 32];
    __shared__ unsigned int hist[256];
    __shared__ unsigned int words[FT / 32];
    __shared__ unsigned long long s_prefix;
    __shared__ unsigned int s_rank, s_cnt_eq;
    __shared__ int s_last, s_count, s_ncand;
    __shared__ double s_sd, s_sd2;

    const T* x = data + (long long)blockIdx.x * stride;
    spx_features* o = out + blockIdx.x;
    int* pk = peaks ? peaks + (long long)blockIdx.x * peaks_cap : nullptr;
    const int tid = threadIdx.x;

    // ---- pass 1: max / argmax (first occurrence), mean, flatness sums (classifier.py:46,183-189)
    // np.max / np.argmax: the first NaN wins over everything; otherwise the first index of the largest value.  A thread
    // takes its first bin unconditionally, so a row of -inf gives argmax 0.
    double vmax = -INFINITY;
    int imax = 0x7fffffff;
    double s1 = 0.0, slog = 0.0, slin = 0.0;
    for (int i = tid; i < n; i += FT) {
        const double v = (double)x[i];
        if (imax == 0x7fffffff || (vmax == vmax && !(v <= vmax))) { vmax = v; imax = i; }
        s1 += v;
        // p = max(10^(v/10), 1e-15) and ln p (classifier.py:185-187): one exp; ln p is v ln(10)/10 unless clipped
        const double lnp = v * 0.23025850929940456840;   // ln(10)/10
        double p = exp(lnp);
        const bool clipped = p < 1e-15;
        p = clipped ? 1e-15 : p;
        slog += clipped ? -34.538776394910684 : lnp;      // ln(1e-15)
        slin += p;
    }
    // one combined block reduction: exact maximum (order-preserving 64-bit key), then first index of it, and the sums
    const unsigned long long kmax = block_max_u64(key_of(vmax), shu);
    const double peak = val_of(kmax);
    const bool is_max = vmax == peak || (vmax != vmax && peak != peak);
    const int argmax = (int)block_min_ll(is_max ? (long long)imax : (long long)0x7fffffff, shl);
    double sums[3] = {s1, slog, slin};
    block_sum3(sums, shd3);
    const double sum_x = sums[0], sum_log = sums[1], sum_lin = sums[2];
    const double mu = sum_x / (double)n;

    // ---- pass 2: variance + occupied-bandwidth edges (classifier.py:163-170, 18-23)
    const double thr3 = __dsub_rn(peak, opts.drop_db[0]), thr10 = __dsub_rn(peak, opts.drop_db[1]);
    const double thr20 = __dsub_rn(peak, opts.drop_db[2]);
    double s2 = 0.0;
    int f3 = 0x7fffffff, l3 = -1, f10 = 0x7fffffff, l10 = -1, f20 = 0x7fffffff, l20 = -1, fs = 0x7fffffff, ls = -1;
    for (int i = tid; i < n; i += FT) {
        const double v = (double)x[i];
        const double d = v - mu;
        s2 += d * d;
        if (v >= thr3) { f3 = min(f3, i); l3 = max(l3, i); }
        if (v >= thr10) { f10 = min(f10, i); l10 = max(l10, i); }
        if (v >= thr20) { f20 = min(f20, i); l20 = max(l20, i); }
        if (v > thr20) { fs = min(fs, i); ls = max(ls, i); }
    }
    const double var = block_sum(s2, shd) / (double)n;
    const double sd = sqrt(var);
    {
        // eight integer min/max in one pass: minima as they are, maxima negated
        int mm[8] = {f3, f10, f20, fs, -l3, -l10, -l20, -ls};
        block_min8(mm, shi8);
        f3 = mm[0]; f10 = mm[1]; f20 = mm[2]; fs = mm[3];
        l3 = -mm[4]; l10 = -mm[5]; l20 = -mm[6]; ls = -mm[7];
    }

    // ---- pass 3: kurtosis (classifier.py:191-198); a NaN sigma (any non-finite bin) gives NaN, as `if sd < 1e-9` does
    double kurt = 0.0;
    if (!(sd < 1e-9)) {
        double s4 = 0.0;
        for (int i = tid; i < n; i += FT) {
            const double z = ((double)x[i] - mu) / sd;
            const double z2 = z * z;
            s4 += z2 * z2;
        }
        kurt = block_sum(s4, shd) / (double)n;
    }

    // ---- radix select: order statistics lo = floor(0.2 (n-1)) and lo+1 (np.percentile 'linear', :181)
    const double virt = __dmul_rn((double)(n - 1), 0.2);
    const int lo = (int)floor(virt);
    const double gamma = __dsub_rn(virt, (double)lo);
    if (tid == 0) { s_prefix = 0ull; s_rank = (unsigned int)lo; }
    unsigned long long mask = 0ull;
    for (int shift = 56; shift >= 0; shift -= 8) {
        if (tid < 256) hist[tid] = 0u;
        __syncthreads();
        const unsigned long long prefix = s_prefix;
        // histogram of the current digit, warp-aggregated: the first passes see only a handful of distinct digits
        // (same sign / exponent), which would serialise thousands of shared-memory atomics on one address
        for (int i0 = 0; i0 < n; i0 += FT) {
            const int i = i0 + tid;
            unsigned int d = 0xffffffffu;
            if (i < n) {
                const unsigned long long k = key_of((double)x[i]);
                if ((k & mask) == prefix) d = (unsigned int)(k >> shift) & 0xffu;
            }
            const unsigned int peers = __match_any_sync(0xffffffffu, d);
            if (d != 0xffffffffu && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[d], (unsigned int)__popc(peers));
        }
        __syncthreads();
        if (tid < 32) {
            // warp-parallel search of the digit that contains rank r: 8 bins per lane + shuffle scan
            const unsigned int r = s_rank;
            unsigned int h[8], mine = 0u;
#pragma unroll
            for (int q = 0; q < 8; ++q) { h[q] = hist[tid * 8 + q]; mine += h[q]; }
            unsigned int incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
                if (tid >= o) incl += t;
            }
            const unsigned int excl = incl - mine;
            const bool here = r >= excl && r < incl;   // exactly one lane (total count > r)
            if (here) {
                unsigned int cum = excl;
                int q = 0;
                for (; q < 7; ++q) {
                    if (r < cum + h[q]) break;
                    cum += h[q];
                }
                s_rank = r - cum;
                s_cnt_eq = h[q];
                s_prefix = prefix | ((unsigned long long)(tid * 8 + q) << shift);
            }
        }
        mask |= 0xffull << shift;
        __syncthreads();
        if (s_cnt_eq == 1u && shift > 0) {
            // a single element carries this prefix: it IS the order statistic; fetch its remaining digits directly
            const unsigned long long prefix1 = s_prefix;
            __syncthreads();
            for (int i = tid; i < n; i += FT) {
                const unsigned long long k = key_of((double)x[i]);
                if ((k & mask) == prefix1) s_prefix = k;
            }
            if (tid == 0) s_rank = 0u;
            __syncthreads();
            break;
        }
    }
    const unsigned long long klo = s_prefix;
    const double vlo = val_of(klo);
    double vhi = vlo;
    if (lo + 1 < n && !(s_rank + 1u < s_cnt_eq)) {
        // next distinct value: smallest key greater than klo
        long long best = LLONG_MAX;
        for (int i = tid; i < n; i += FT) {
            const unsigned long long k = key_of((double)x[i]);
            if (k > klo) { const long long kk = (long long)(k >> 1); best = kk < best ? kk : best; }
        }
        const long long b1 = block_min_ll(best, shl);
        long long low = 2;
        for (int i = tid; i < n; i += FT) {
            const unsigned long long k = key_of((double)x[i]);
            if (k > klo && (long long)(k >> 1) == b1) { const long long lb = (long long)(k & 1ull); low = lb < low ? lb : low; }
        }
        low = block_min_ll(low, shl);
        vhi = val_of(((unsigned long long)b1 << 1) | (unsigned long long)low);
    }
    // numpy _lerp: a + (b-a)*t, or b - (b-a)*(1-t) when t >= 0.5 (no fused multiply-add); also for n == 1, where
    // a == b and an infinite a gives NaN as in numpy.  np.percentile is NaN when any bin is NaN, i.e. when the peak is.
    const double diff = __dsub_rn(vhi, vlo);
    double nf = __dadd_rn(vlo, __dmul_rn(diff, gamma));
    if (gamma >= 0.5) nf = __dsub_rn(vhi, __dmul_rn(diff, __dsub_rn(1.0, gamma)));
    if (peak != peak) nf = peak;

    const double snr = __dsub_rn(peak, nf);
    // max(nf + 5, peak - 0.9*snr + 5)  (classifier.py:53), as Python's max: the second only when it is greater, so a
    // NaN second term (one +inf bin: inf - 0.9 inf) leaves nf + 5
    const double thr_a = __dadd_rn(nf, 5.0);
    const double thr_b = __dadd_rn(__dsub_rn(peak, __dmul_rn(0.9, snr)), 5.0);
    double thr = thr_b > thr_a ? thr_b : thr_a;
    if (opts.use_peak_threshold) thr = opts.peak_threshold_db;
    const int min_dist = opts.min_distance_bins > 0 ? opts.min_distance_bins : max(3, n / 300);

    // ---- peaks: strict interior local maxima above thr, greedy left-to-right thinning (:200-212)
    if (tid == 0) { s_last = -min_dist; s_count = 0; s_ncand = 0; s_sd = 0.0; s_sd2 = 0.0; }
    __syncthreads();
    for (int base = 0; base < n; base += FT) {
        const int i = base + tid;
        bool c = false;
        if (i >= 1 && i < n - 1) {
            const double v = (double)x[i];
            c = v > thr && v > (double)x[i - 1] && v > (double)x[i + 1];
        }
        const unsigned int b = __ballot_sync(0xffffffffu, c);
        if ((tid & 31) == 0) words[tid >> 5] = b;
        __syncthreads();
        if (tid == 0) {
            int last = s_last, cnt = s_count, nc = s_ncand;
            double sdv = s_sd, sd2v = s_sd2;
            for (int w = 0; w < FT / 32; ++w) {
                unsigned int m = words[w];
                while (m) {
                    const int bit = __ffs(m) - 1;
                    m &= m - 1;
                    const int idx = base + 32 * w + bit;
                    ++nc;
                    if ((long long)idx - last >= min_dist) {   // 64-bit: last starts at -min_dist, up to -INT32_MAX
                        if (cnt > 0) { const double d = (double)(idx - last); sdv += d; sd2v += d * d; }
                        if (pk && cnt < peaks_cap) pk[cnt] = idx;
                        ++cnt;
                        last = idx;
                    }
                }
            }
            s_last = last; s_count = cnt; s_ncand = nc; s_sd = sdv; s_sd2 = sd2v;
        }
        __syncthreads();
    }

    if (tid == 0) {
        o->n = n;
        o->argmax = argmax;
        o->peak_db = peak;
        o->noise_floor_db = nf;
        o->snr_db = snr;
        o->adaptive_thr = thr;
        o->p20_lo = vlo;
        o->p20_hi = vhi;
        o->min_distance_bins = min_dist;
        o->first_3db = l3 < 0 ? -1 : f3;    o->last_3db = l3;
        o->first_10db = l10 < 0 ? -1 : f10; o->last_10db = l10;
        o->first_20db = l20 < 0 ? -1 : f20; o->last_20db = l20;
        o->simple_first = ls < 0 ? -1 : fs; o->simple_last = ls;
        const double geo = exp(sum_log / (double)n);
        const double ari = sum_lin / (double)n;
        double fl = geo / ari;
        fl = fl < 0.0 ? 0.0 : (fl > 1.0 ? 1.0 : fl);
        o->flatness = fl;
        o->kurtosis = kurt;
        o->mean_db = mu;
        o->std_db = sd;
        o->n_candidates = s_ncand;
        o->peak_count = s_count;
        double sp = 0.0;
        if (s_count >= 3) {
            const double m = (double)(s_count - 1);
            const double mean_d = s_sd / m;
            const double v = s_sd2 / m - mean_d * mean_d;
            sp = v > 0.0 ? sqrt(v) : 0.0;
        }
        o->peak_spacing_std_bins = sp;
        o->peaks_stored = pk ? (s_count < peaks_cap ? s_count : peaks_cap) : 0;
        o->reserved = 0;
    }
}

// features_kernel over `batch` spectra of n bins, `stride` apart, in float32 (dtype 0) or float64 (dtype 1, checked by the
// caller); NULL user_opts: the reference's options
int features_launch(const void* in, int dtype, int n, int batch, long long stride, spx_features* out, int* peaks,
                           int peaks_cap, const spx_feature_opts* user_opts, cudaStream_t st) {
    spx_feature_opts opts;
    memset(&opts, 0, sizeof(opts));
    opts.drop_db[0] = 3.0; opts.drop_db[1] = 10.0; opts.drop_db[2] = 20.0;
    if (user_opts) opts = *user_opts;
    if (dtype)
        features_kernel<double><<<batch, FT, 0, st>>>((const double*)in, n, stride, out, peaks, peaks_cap, opts);
    else
        features_kernel<float><<<batch, FT, 0, st>>>((const float*)in, n, stride, out, peaks, peaks_cap, opts);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

}  // namespace spx

using namespace spx;

extern "C" int spx_classify_features(int32_t device, int32_t mem, const void* power_db, int32_t dtype, int32_t n,
                                     int32_t batch, int64_t stride, spx_features* out, int32_t* peaks,
                                     int32_t peaks_cap, const spx_feature_opts* user_opts, void* stream) {
    if (!out) return spx_set_error(SPX_E_INVALID, "out is NULL");
    if (batch < 0 || n < 0) return spx_set_error(SPX_E_INVALID, "negative size");
    if (dtype != 0 && dtype != 1) return spx_set_error(SPX_E_INVALID, "dtype must be 0 (float32) or 1 (float64)");
    if (batch == 0) return SPX_OK;
    if (n == 0) {  // empty spectrum: the host layer answers "No Data" (classifier.py:41-42)
        memset(out, 0, sizeof(spx_features) * (size_t)batch);
        return SPX_OK;
    }
    if (!power_db) return spx_set_error(SPX_E_INVALID, "power_db is NULL");
    if (batch > 1 && stride < n) return spx_set_error(SPX_E_INVALID, "stride < n");
    if (peaks && peaks_cap < 1) peaks = nullptr;
    DeviceCtx* ctx;
    SPX_TRY(device_ctx(device, &ctx));
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaStream_t st = (mem == SPX_MEM_DEVICE && stream) ? (cudaStream_t)stream : ctx->st;
    const void* d_in = power_db;
    long long d_stride = stride;
    size_t in_bytes = 0;
    if (mem == SPX_MEM_HOST) {
        if (batch == 1) d_stride = n;
        in_bytes = ((size_t)(batch - 1) * (size_t)d_stride + (size_t)n) * (dtype ? 8 : 4);
    }
    const size_t out_bytes = sizeof(spx_features) * (size_t)batch;
    const size_t pk_bytes = peaks ? sizeof(int) * (size_t)batch * (size_t)peaks_cap : 0;
    void* part[3];   // staged input (host memory only), results, peaks
    SPX_TRY(ctx->carve({in_bytes, out_bytes, pk_bytes}, part));
    if (mem == SPX_MEM_HOST) {
        SPX_CUDA(cudaMemcpyAsync(part[0], power_db, in_bytes, cudaMemcpyHostToDevice, st));
        d_in = part[0];
    }
    int* d_pk = peaks ? (int*)part[2] : nullptr;
    SPX_TRY(features_launch(d_in, dtype, n, batch, d_stride, (spx_features*)part[1], d_pk, peaks_cap, user_opts, st));
    SPX_CUDA(cudaMemcpyAsync(out, part[1], out_bytes, cudaMemcpyDeviceToHost, st));
    if (peaks) SPX_CUDA(cudaMemcpyAsync(peaks, d_pk, pk_bytes, cudaMemcpyDeviceToHost, st));
    SPX_CUDA(cudaStreamSynchronize(st));
    return SPX_OK;
}

extern "C" int spx_classify_features_dev(int32_t device, const void* power_db_dev, int32_t dtype, int32_t n, int32_t batch,
                                         int64_t stride, spx_features* out_dev, int32_t* peaks_dev, int32_t peaks_cap,
                                         const spx_feature_opts* user_opts, void* stream) {
    if (!out_dev || !power_db_dev) return spx_set_error(SPX_E_INVALID, "NULL argument");
    if (batch < 1 || n < 1) return spx_set_error(SPX_E_INVALID, "batch and n must be positive");
    if (dtype != 0 && dtype != 1) return spx_set_error(SPX_E_INVALID, "dtype must be 0 (float32) or 1 (float64)");
    if (batch > 1 && stride < n) return spx_set_error(SPX_E_INVALID, "stride < n");
    if (peaks_dev && peaks_cap < 1) peaks_dev = nullptr;
    SPX_CUDA(cudaSetDevice(device));
    return features_launch(power_db_dev, dtype, n, batch, stride, out_dev, peaks_dev, peaks_cap, user_opts, (cudaStream_t)stream);
}
