// spx_chan.cu -- polyphase filter-bank channelizer (DESIGN.md section 4, K10) and its C ABI (spx_chan_*).
//
//   y_j[m] = sum_k h[k] x[mD + T-1-k] exp(-2 pi i (j - M/2) (first_sample + mD + T-1-k) / M),   j = 0 .. M-1
//
// = the M-point DFT (fftshift order) of the fold v_m[r] over the tap classes r = global sample index mod M
// (spx_chan_device.cuh).  A CTA runs F frames (outputs) at a time, M/16 threads each (F M / 16 <= 256 threads), and
// owns a contiguous run of sub-tiles of F outputs.  Each thread folds its 16 classes, then the frame runs the STFT's
// Stockham passes through one exchange buffer; the bins are transposed through that buffer into [M][F] and leave as runs
// of F outputs per channel.  The input reaches the fold in one of two ways:
//   ring:    a shared-memory ring of F D + max(T - D, 0) samples (scaled to float2 once as they arrive) that holds the
//            windows of a whole sub-tile, so a CTA reads its T - D halo once, not once per sub-tile, and HBM is read about
//            once per sample.  Used when that ring fits with the full 256 threads.
//   blocked: for longer windows, each sub-tile streams its windows through a shared-memory stage in blocks of TB window
//            offsets ((F - 1) D + TB samples a block); the partial folds stay in registers from block to block, so every
//            class is summed in the same order as in the ring mode.  A sample is read about T / (F D) times, from L2.
// The reversed taps sit in shared memory when they fit next to the ring, else they are read from global memory.
#include <mutex>
#include <new>

#include "spx_chan_device.cuh"
#include "spx_fir.h"
#include "spx_internal.h"
#include "spx_tables.h"

namespace spx {

constexpr int CHAN_MAX_THREADS = 256;
constexpr int CHAN_MIN_M = 16, CHAN_MAX_M = 4096;

struct ChanParams {
    const void* in;
    long long L;               // samples of the call
    unsigned long long n0;     // global index of sample 0 (first_sample)
    const float* taps;         // g[j] = h[T - 1 - j], float32 (global)
    const float2* tw;          // twiddle table of the M-point FFT (build_twiddles)
    float2* out;               // [M][out_stride]
    long long out_stride;
    long long n_out;
    long long n_sub;           // sub-tiles of F outputs
    float scale;
    int T, D, F, ring, taps_smem;
    int tb;                    // blocked mode: window offsets per block (0: ring mode)
};

template <int FMT>
__device__ inline float2 chan_load(const void* in, long long n, float scale) {
    float xr, xi;
    if (FMT == SPX_FMT_CI16) {
        const short2 v = __ldg(reinterpret_cast<const short2*>(in) + n);
        xr = (float)v.x;
        xi = (float)v.y;
    } else {
        const float* f = reinterpret_cast<const float*>(in) + 2 * n;
        xr = __ldg(f);
        xi = __ldg(f + 1);
    }
    return make_float2(ddc_mul(xr, scale), ddc_mul(xi, scale));
}

// samples n_cta + [lo, hi) of the call into the ring (slot = r mod ring); samples past the call's end are zero
template <int FMT>
__device__ inline void chan_fill(const ChanParams& p, float2* ring, long long n_cta, long long lo, long long hi) {
    constexpr int U = 4;
    const int nt = blockDim.x;
    long long r = lo + threadIdx.x;
    int slot = (int)(r % p.ring);
    for (; r < hi; r += U * nt) {
        float2 x[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long rr = r + u * nt, n = n_cta + rr;
            x[u] = make_float2(0.f, 0.f);
            if (rr < hi && n < p.L) x[u] = chan_load<FMT>(p.in, n, p.scale);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (r + u * nt < hi) ring[slot] = x[u];
            slot += nt;
            if (slot >= p.ring) slot -= p.ring;
        }
    }
}

// passes S .. P-1 of the frame's FFT through the exchange buffer (pass S - 1's result in v)
template <int M, int S>
__device__ __forceinline__ void chan_passes(float2* v, int ft, float2* fb, const float2* tw) {
    if constexpr (S < plan_passes(M)) {
        pass_store_smem<M, S - 1>(v, ft, fb);
        __syncthreads();
        chan_pass<M, S>(v, ft, fb, tw);
        __syncthreads();
        chan_passes<M, S + 1>(v, ft, fb, tw);
    }
}

template <int FMT, int M>
__global__ void __launch_bounds__(CHAN_MAX_THREADS, 2) chan_kernel(const ChanParams p) {
    constexpr int TPF = M / 16, P = plan_passes(M), R = plan_radix(M, P - 1), NB = 16 / R;
    extern __shared__ float4 chan_smem[];
    float2* buf = reinterpret_cast<float2*>(chan_smem);            // [F][padded_size(M)]: exchange, then the [M][F] tile
    float2* ring = buf + (size_t)p.F * padded_size(M);
    float* gs = reinterpret_cast<float*>(ring + p.ring);
    const int tid = threadIdx.x, f = tid / TPF, ft = tid % TPF, F = p.F;
    const float* g = p.taps;
    if (p.taps_smem) {
        for (int i = tid; i < p.T; i += blockDim.x) gs[i] = p.taps[i];
        g = gs;
    }
    float2* fb = buf + (size_t)f * padded_size(M);
    const long long sb0 = (long long)blockIdx.x * p.n_sub / gridDim.x;
    const long long sb1 = (long long)(blockIdx.x + 1) * p.n_sub / gridDim.x;
    const long long n_cta = sb0 * F * (long long)p.D;   // call index of the CTA's sample 0
    long long filled = 0;
    for (long long k = sb0; k < sb1; ++k) {
        const long long kk = k - sb0;
        const long long m = k * F + f;   // this frame's output
        const unsigned cls0 = chan_cls0(p.n0, m, p.D, M);
        float2 v[16];
#pragma unroll
        for (int t = 0; t < 16; ++t) v[t] = make_float2(0.f, 0.f);
        if (p.tb == 0) {
            const long long hi = (kk + 1) * F * (long long)p.D + p.T - p.D;
            chan_fill<FMT>(p, ring, n_cta, filled, hi);
            filled = hi;
            __syncthreads();
            const long long rel = (kk * F + f) * (long long)p.D;
            chan_fold<M>(v, ft, g, 0, p.T, ring, p.ring, (int)(rel % p.ring), cls0);
        } else {
            const long long n_sub0 = k * F * (long long)p.D;   // call index of the sub-tile's first window
            for (int j_lo = 0; j_lo < p.T; j_lo += p.tb) {
                const int j_hi = p.T - j_lo < p.tb ? p.T : j_lo + p.tb;
                __syncthreads();   // the previous block's folds are done with the stage
                chan_fill<FMT>(p, ring, n_sub0 + j_lo, 0, (long long)(F - 1) * p.D + (j_hi - j_lo));
                __syncthreads();
                chan_fold<M>(v, ft, g, j_lo, j_hi, ring, p.ring, f * p.D - j_lo, cls0);
            }
        }
        pass_dft<M, 0>(v);
        chan_passes<M, 1>(v, ft, fb, p.tw);   // ends with a barrier when P > 1: every exchange read is done
        // transpose: channel j of frame f -> buf[j F + f]
#pragma unroll
        for (int u = 0; u < NB; ++u)
#pragma unroll
            for (int t = 0; t < R; ++t) buf[chan_of<M>(ft, u, t) * F + f] = v[u * R + t];
        __syncthreads();
        const long long mk = k * F;
        const int nf = (int)(p.n_out - mk < F ? p.n_out - mk : F);
        for (int idx = tid; idx < M * F; idx += blockDim.x) {
            const int j = idx / F, c = idx - j * F;
            if (c < nf) p.out[j * p.out_stride + mk + c] = buf[idx];
        }
        __syncthreads();   // the tile is read before the next frame's exchange writes buf
    }
}

// ------------------------------------------------------------------ launch geometry
struct ChanLaunch {
    int F, threads, ring, taps_smem, tb;
    size_t smem;
};

static size_t chan_smem_bytes(int M, int F, int ring, int T, bool taps_smem) {
    return (size_t)F * padded_size(M) * 8 + (size_t)ring * 8 + (taps_smem ? (size_t)((T + 3) & ~3) * 4 : 0);
}

// F = 256 / (M / 16) frames per CTA.  Ring mode when the ring of F D + max(T - D, 0) samples fits one CTA; else blocked
// mode with the largest block of TB window offsets (a multiple of M) whose stage leaves two CTAs per SM.  Taps in shared
// memory when they fit too and two CTAs per SM remain.
static void chan_plan_launch(int M, int T, int D, int max_smem, ChanLaunch* out) {
    const size_t two = (size_t)max_smem / 2 - 1024;   // two CTAs per SM (1 KB reserved per CTA)
    ChanLaunch L;
    L.F = CHAN_MAX_THREADS / (M / 16);
    L.threads = CHAN_MAX_THREADS;
    L.ring = L.F * D + (T > D ? T - D : 0);
    L.tb = 0;
    if (chan_smem_bytes(M, L.F, L.ring, T, false) > (size_t)max_smem) {
        const size_t fixed = chan_smem_bytes(M, L.F, (L.F - 1) * D, T, false);
        long long tb = fixed < two ? (long long)((two - fixed) / 8) / M * M : 0;
        if (tb < M) tb = M;
        if (tb > T) tb = T;
        L.tb = (int)tb;
        L.ring = (L.F - 1) * D + L.tb;   // at most 34 KB of exchange buffer + 32 KB + M samples: always fits one CTA
    }
    const size_t with_taps = chan_smem_bytes(M, L.F, L.ring, T, true);
    L.taps_smem = with_taps <= two;
    L.smem = chan_smem_bytes(M, L.F, L.ring, T, L.taps_smem);
    *out = L;
}

template <int FMT>
static const void* chan_kernel_ptr(int M) {
    switch (M) {
        case 16: return (const void*)chan_kernel<FMT, 16>;
        case 32: return (const void*)chan_kernel<FMT, 32>;
        case 64: return (const void*)chan_kernel<FMT, 64>;
        case 128: return (const void*)chan_kernel<FMT, 128>;
        case 256: return (const void*)chan_kernel<FMT, 256>;
        case 512: return (const void*)chan_kernel<FMT, 512>;
        case 1024: return (const void*)chan_kernel<FMT, 1024>;
        case 2048: return (const void*)chan_kernel<FMT, 2048>;
        default: return (const void*)chan_kernel<FMT, 4096>;
    }
}

}  // namespace spx

using namespace spx;

struct spx_chan : FirHandle {
    int n_channels = 0, occ = 1;
    float2* d_tw = nullptr;     // M-point twiddle table
    ChanLaunch launch{};
};

namespace spx {

// K10 over samples [0, L) of `in` (device), global index of sample 0 = n0, outputs -> out[M][out_stride] (device)
static int chan_launch(spx_chan* h, const void* in, long long L, unsigned long long n0, float2* out, long long out_stride,
                       cudaStream_t st) {
    const long long n_out = h->out_count(L);
    if (n_out <= 0) return SPX_OK;
    const ChanLaunch& G = h->launch;
    ChanParams p;
    p.in = in;
    p.L = L;
    p.n0 = n0;
    p.taps = h->d_taps;
    p.tw = h->d_tw;
    p.out = out;
    p.out_stride = out_stride;
    p.n_out = n_out;
    p.n_sub = (n_out + G.F - 1) / G.F;
    p.scale = h->in_scale;
    p.T = h->n_taps;
    p.D = h->decim;
    p.F = G.F;
    p.ring = G.ring;
    p.taps_smem = G.taps_smem;
    p.tb = G.tb;
    const long long cap = (long long)h->occ * (h->sm_count > 0 ? h->sm_count : 148);
    const unsigned grid = (unsigned)(p.n_sub < cap ? p.n_sub : cap);
    void* args[] = {&p};
    SPX_CUDA(cudaLaunchKernel(h->kern, dim3(grid), dim3(G.threads), args, G.smem, st));
    return SPX_OK;
}

// Host memory: pieces of about piece_bytes of input (FirHandle::host_pieces).  Piece k's [M][per] block goes to one of
// two device buffers and drains into the caller's [M][out_stride] rows with one 2-D copy.
static int chan_exec_host(spx_chan* h, const void* in, long long n_out, unsigned long long n0, float2* out,
                          long long out_stride, int64_t* h2d_out, int64_t* d2h_out) {
    const int M = h->n_channels;
    const long long per = h->piece_outputs(n_out);
    const size_t block = (size_t)M * (size_t)per;
    SPX_TRY(h->st_out.reserve(2 * block * 8));
    float2* d_out[2] = {(float2*)h->st_out.ptr, (float2*)h->st_out.ptr + block};
    auto launch = [&](const void* d_in, long long n, long long a, long long, long long, int b, cudaStream_t st) {
        return chan_launch(h, d_in, n, n0 + (unsigned long long)a, d_out[b], per, st);
    };
    auto drain = [&](long long m0, long long nm, int b, cudaStream_t st, long long* bytes) {
        SPX_CUDA(cudaMemcpy2DAsync(out + m0, (size_t)out_stride * 8, d_out[b], (size_t)per * 8, (size_t)nm * 8, (size_t)M,
                                   cudaMemcpyDeviceToHost, st));
        *bytes = nm * 8 * (long long)M;
        return SPX_OK;
    };
    return h->host_pieces(in, n_out, per, true, launch, drain, h2d_out, d2h_out);
}

// the twiddle table, and the occupancy that caps the grid (after FirHandle::setup raised the kernel's limit)
static int chan_setup(spx_chan* h) {
    SPX_TRY(upload(&h->d_tw, build_twiddles(h->n_channels)));
    SPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&h->occ, h->kern, h->launch.threads, h->launch.smem));
    if (h->occ < 1) h->occ = 1;
    return SPX_OK;
}

}  // namespace spx

extern "C" {

int spx_chan_create(spx_chan** out, const spx_chan_config* cfg) {
    if (!out || !cfg) return spx_set_error(SPX_E_INVALID, "NULL argument");
    *out = nullptr;
    if (cfg->struct_size != sizeof(spx_chan_config))
        return spx_set_error(SPX_E_INVALID, "spx_chan_config.struct_size %u != %zu", cfg->struct_size, sizeof(spx_chan_config));
    const int M = cfg->n_channels;
    if (M < CHAN_MIN_M || M > CHAN_MAX_M || (M & (M - 1)))
        return spx_set_error(SPX_E_INVALID, "n_channels %d must be a power of two in [%d, %d]", M, CHAN_MIN_M, CHAN_MAX_M);
    if (cfg->decim != M && cfg->decim != M / 2)
        return spx_set_error(SPX_E_INVALID, "decim %d must be n_channels (%d) or n_channels / 2", cfg->decim, M);
    if (cfg->n_taps < 1 || cfg->n_taps > 32 * M)
        return spx_set_error(SPX_E_INVALID, "n_taps %d must be in [1, 32 n_channels = %d]", cfg->n_taps, 32 * M);
    if (!cfg->taps) return spx_set_error(SPX_E_INVALID, "taps is NULL");
    if (cfg->in_fmt != SPX_FMT_CF32 && cfg->in_fmt != SPX_FMT_CI16) return spx_set_error(SPX_E_INVALID, "unknown in_fmt %d", cfg->in_fmt);
    int max_smem = 0, sms = 0;
    SPX_TRY(fir_device(cfg->device, &max_smem, &sms));
    ChanLaunch launch;
    chan_plan_launch(M, cfg->n_taps, cfg->decim, max_smem, &launch);
    spx_chan* h = new (std::nothrow) spx_chan();
    if (!h) return spx_set_error(SPX_E_NOMEM, "out of host memory");
    h->n_channels = M;
    h->launch = launch;
    const void* kern = cfg->in_fmt == SPX_FMT_CI16 ? chan_kernel_ptr<SPX_FMT_CI16>(M) : chan_kernel_ptr<SPX_FMT_CF32>(M);
    int rc = h->setup(*cfg, kern, max_smem, sms);
    if (rc == SPX_OK) rc = chan_setup(h);
    if (rc != SPX_OK) {
        spx_chan_destroy(h);
        return rc;
    }
    *out = h;
    return SPX_OK;
}

int spx_chan_destroy(spx_chan* h) {
    if (!h) return SPX_OK;
    h->release();
    if (h->d_tw) cudaFree(h->d_tw);
    delete h;
    return SPX_OK;
}

int spx_chan_sync(spx_chan* h) {
    if (!h) return spx_set_error(SPX_E_INVALID, "channelizer is NULL");
    return h->sync();
}

int spx_chan_exec(spx_chan* h, int32_t mem, const void* in, int64_t n_samples, int64_t first_sample, float* out,
                  int64_t out_stride, int64_t* n_out, int64_t* h2d_bytes_out, int64_t* d2h_bytes_out, void* stream) {
    if (!h) return spx_set_error(SPX_E_INVALID, "channelizer is NULL");
    long long M = 0;
    std::unique_lock<std::mutex> lock;
    SPX_TRY(h->exec_begin(mem, in, n_samples, first_sample, out, 8, &M, n_out, h2d_bytes_out, d2h_bytes_out, &lock));
    if (M == 0) return SPX_OK;
    if (out_stride < M) return spx_set_error(SPX_E_INVALID, "out_stride %lld < n_out %lld", (long long)out_stride, M);
    if (mem == SPX_MEM_DEVICE)
        return chan_launch(h, in, n_samples, (unsigned long long)first_sample, (float2*)out, out_stride,
                           stream ? (cudaStream_t)stream : h->s_compute);
    return chan_exec_host(h, in, M, (unsigned long long)first_sample, (float2*)out, out_stride, h2d_bytes_out, d2h_bytes_out);
}

}  // extern "C"
