// spx_ddc.cu -- digital down-converter: NCO mix + decimating FIR (DESIGN.md section 4, K9) and its C ABI (spx_ddc_*).
//
//   y[m] = sum_k h[k] mix[mD + T - 1 - k],   mix[n] = x[n] in_scale exp(-2 pi i ((first_sample + n) inc mod 2^64) / 2^64)
//
// A CTA owns a contiguous run of sub-tiles of SUB outputs.  Its mixed input lives in a shared-memory ring of
// SUB D + T - 1 float2 samples: each sub-tile mixes the SUB D samples it adds (one NCO evaluation per sample, strategy
// (a) of DESIGN.md K9), so a CTA mixes its T - 1 halo samples once, not once per sub-tile.  The reversed taps sit in shared
// memory.  A warp computes R = 16 outputs m, m + s, ..., m + 15 s: lane l sums the taps j = l (mod 32) with a register
// window that slides over the outputs (spx_ddc_device.cuh), so one shared load of a sample and one of a tap feed 32
// FMAs.  A reduce-scatter over the lanes leaves output l / 2, component l % 2 in lane l; WR warps that split the tap
// classes of the same outputs are added in a fixed order before the store.
#include <mutex>
#include <new>

#include "spx_ddc_device.cuh"
#include "spx_fir.h"
#include "spx_internal.h"

namespace spx {

constexpr int DDC_THREADS = 256;   // 8 warps
constexpr int DDC_R = 16;          // outputs per warp: 2 R = 32 values, one per lane after the reduce-scatter
constexpr int DDC_MAX_TAPS = 8192;
constexpr size_t DDC_SMEM_TWO_PER_SM = 110u << 10;   // two CTAs per SM (228 KB, 1 KB reserved per CTA)

struct DdcParams {
    const void* in;
    long long L;              // samples of the call
    unsigned long long n0;    // global index of sample 0 (first_sample)
    unsigned long long inc;   // phase increment
    const float* taps;        // g[j] = h[T - 1 - j], float32
    float* out;               // [M][2]
    long long M;
    long long n_sub;          // sub-tiles of the call
    float scale;
    int T, D, sub, ring, taps_pad;
    int s, c, wr, wg;
};

template <int FMT>
__device__ inline void ddc_load(const void* in, long long n, float* xr, float* xi) {
    if (FMT == SPX_FMT_CI16) {
        const short2 v = __ldg(reinterpret_cast<const short2*>(in) + n);
        *xr = (float)v.x;
        *xi = (float)v.y;
    } else {
        const float* f = reinterpret_cast<const float*>(in) + 2 * n;
        *xr = __ldg(f);
        *xi = __ldg(f + 1);
    }
}

// mix CTA-relative samples [lo, hi) into the ring (slot = r mod ring); samples past the call's end are zero
template <int FMT>
__device__ inline void ddc_mix_range(const DdcParams& p, float2* ring, long long n_cta, long long lo, long long hi) {
    long long r = lo + threadIdx.x;
    int slot = (int)(r % p.ring);
    constexpr int U = 4;
    for (; r < hi; r += U * DDC_THREADS) {
        float xr[U], xi[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long rr = r + u * DDC_THREADS, n = n_cta + rr;
            xr[u] = 0.f;
            xi[u] = 0.f;
            if (rr < hi && n < p.L) ddc_load<FMT>(p.in, n, &xr[u], &xi[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long rr = r + u * DDC_THREADS;
            if (rr < hi) {
                const long long n = n_cta + rr;
                float re, im;
                ddc_mix(ddc_mul(xr[u], p.scale), ddc_mul(xi[u], p.scale), ddc_phase(p.n0 + (unsigned long long)n, p.inc), &re,
                        &im);
                ring[slot] = make_float2(re, im);
            }
            slot += DDC_THREADS;
            if (slot >= p.ring) slot -= p.ring;
        }
    }
}

// one step t of a lane's sliding window: load element t + R - 1 into w[(K + R - 1) % R], then 2 R FMAs
template <int K>
__device__ __forceinline__ void ddc_step(float (&ar)[DDC_R], float (&ai)[DDC_R], float (&wre)[DDC_R], float (&wim)[DDC_R],
                                         const float2* ring, int& slot, int step, int ring_n, float gv) {
    const float2 v = ring[slot];
    wre[(K + DDC_R - 1) % DDC_R] = v.x;
    wim[(K + DDC_R - 1) % DDC_R] = v.y;
    slot += step;
    if (slot >= ring_n) slot -= ring_n;
#pragma unroll
    for (int i = 0; i < DDC_R; ++i) {
        ar[i] = fmaf(gv, wre[(K + i) % DDC_R], ar[i]);
        ai[i] = fmaf(gv, wim[(K + i) % DDC_R], ai[i]);
    }
}

template <int... Ks>
struct DdcSteps;
template <>
struct DdcSteps<> {
    template <bool GUARD>
    __device__ __forceinline__ static void run(float (&)[DDC_R], float (&)[DDC_R], float (&)[DDC_R], float (&)[DDC_R],
                                               const float2*, int&, int, int, const float*, int, int) {}
};
template <int K, int... Ks>
struct DdcSteps<K, Ks...> {
    // taps t0 + K, t0 + K + 1, ... (GUARD: only those < n)
    template <bool GUARD>
    __device__ __forceinline__ static void run(float (&ar)[DDC_R], float (&ai)[DDC_R], float (&wre)[DDC_R],
                                               float (&wim)[DDC_R], const float2* ring, int& slot, int step, int ring_n,
                                               const float* gp, int t0, int n) {
        if (GUARD && t0 + K >= n) return;
        ddc_step<K>(ar, ai, wre, wim, ring, slot, step, ring_n, gp[(t0 + K) * step]);
        DdcSteps<Ks...>::template run<GUARD>(ar, ai, wre, wim, ring, slot, step, ring_n, gp, t0, n);
    }
};
using DdcAllSteps = DdcSteps<0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15>;
static_assert(DDC_R == 16, "DdcAllSteps lists R steps");

template <int FMT>
__global__ void __launch_bounds__(DDC_THREADS, 2) ddc_kernel(const DdcParams p) {
    extern __shared__ float4 ddc_smem[];
    float* g = reinterpret_cast<float*>(ddc_smem);
    float2* ring = reinterpret_cast<float2*>(g + p.taps_pad);
    float* red = reinterpret_cast<float*>(ring + p.ring);   // [wr][sub][2]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < p.T; i += DDC_THREADS) g[i] = p.taps[i];
    const long long sb0 = (long long)blockIdx.x * p.n_sub / gridDim.x;
    const long long sb1 = (long long)(blockIdx.x + 1) * p.n_sub / gridDim.x;
    const long long n_cta = sb0 * p.sub * (long long)p.D;   // call index of the CTA's sample 0
    const int wr = warp % p.wr, wg = warp / p.wr;
    const int groups = p.sub / DDC_R, step = 32 * p.c;
    long long mixed = 0;
    for (long long k = sb0; k <= sb1; ++k) {
        const long long kk = k - sb0;
        if (k < sb1) {
            const long long hi = (kk + 1) * p.sub * (long long)p.D + p.T - 1;
            ddc_mix_range<FMT>(p, ring, n_cta, mixed, hi);
            mixed = hi;
        }
        if (k > sb0) {   // the outputs of the previous sub-tile: warp partials in order of wr
            for (int idx = tid; idx < 2 * p.sub; idx += DDC_THREADS) {
                const long long m = (k - 1) * p.sub + (idx >> 1);
                if (m >= p.M) break;
                float v = red[idx];
                for (int w = 1; w < p.wr; ++w) v = __fadd_rn(v, red[w * 2 * p.sub + idx]);
                p.out[2 * m + (idx & 1)] = v;
            }
        }
        if (k == sb1) break;
        __syncthreads();
        for (int gi = wg; gi < groups; gi += p.wg) {
            const int mm0 = (gi / p.s) * DDC_R * p.s + gi % p.s;
            float ar[DDC_R], ai[DDC_R];
#pragma unroll
            for (int i = 0; i < DDC_R; ++i) ar[i] = ai[i] = 0.f;
            for (int rho = wr; rho < p.c; rho += p.wr) {
                const int n = ddc_lane_taps(p.T, p.c, lane, rho);
                if (n == 0) continue;
                const long long r0 = (kk * p.sub + mm0) * (long long)p.D + 32 * rho + lane;
                int slot = (int)(r0 % p.ring);
                const float* gp = g + 32 * rho + lane;
                float wre[DDC_R], wim[DDC_R];
#pragma unroll
                for (int e = 0; e < DDC_R - 1; ++e) {
                    const float2 v = ring[slot];
                    wre[e] = v.x;
                    wim[e] = v.y;
                    slot += step;
                    if (slot >= p.ring) slot -= p.ring;
                }
                int t0 = 0;
                for (; t0 + DDC_R <= n; t0 += DDC_R)
                    DdcAllSteps::run<false>(ar, ai, wre, wim, ring, slot, step, p.ring, gp, t0, n);
                DdcAllSteps::run<true>(ar, ai, wre, wim, ring, slot, step, p.ring, gp, t0, n);
            }
            // reduce-scatter: value 2 i + comp of every lane, tree pairs (l, l ^ 16), (l, l ^ 8), ... -> lane 2 i + comp
            float v[2 * DDC_R];
#pragma unroll
            for (int i = 0; i < DDC_R; ++i) {
                v[2 * i] = ar[i];
                v[2 * i + 1] = ai[i];
            }
#pragma unroll
            for (int half = 16; half >= 1; half >>= 1) {
                const bool up = (lane & half) != 0;
#pragma unroll
                for (int i = 0; i < half; ++i) {
                    const float send = up ? v[i] : v[i + half];
                    const float keep = up ? v[i + half] : v[i];
                    v[i] = __fadd_rn(keep, __shfl_xor_sync(0xffffffffu, send, half));
                }
            }
            red[(wr * p.sub + mm0 + (lane >> 1) * p.s) * 2 + (lane & 1)] = v[0];
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ launch geometry
struct DdcLaunch {
    DdcGeom G;
    int sub, ring, taps_pad;
    size_t smem;
};

static size_t ddc_smem_bytes(int T, int D, int wr, int sub, int* ring, int* taps_pad) {
    *taps_pad = (T + 3) & ~3;
    *ring = sub * D + T - 1;
    return (size_t)*taps_pad * 4 + (size_t)*ring * 8 + (size_t)wr * sub * 8;
}

// SUB = R max(s, wg) k with the largest k that keeps two CTAs per SM (k = 1 and one CTA per SM when even that is too big)
static int ddc_plan_launch(int T, int D, int max_smem, DdcLaunch* out) {
    DdcLaunch L;
    L.G = ddc_geom(D);
    const int base = DDC_R * (L.G.s > L.G.wg ? L.G.s : L.G.wg);
    int ring, tp;
    if (ddc_smem_bytes(T, D, L.G.wr, base, &ring, &tp) > (size_t)max_smem)
        return spx_set_error(SPX_E_UNSUPPORTED,
                             "decim %d with %d taps needs more shared memory than one CTA has: decimate in two stages "
                             "(a second DDC with shift 0 on the first one's output)", D, T);
    int k = 1;
    while ((long long)base * (k + 1) * D <= 16384 &&
           ddc_smem_bytes(T, D, L.G.wr, base * (k + 1), &ring, &tp) <= DDC_SMEM_TWO_PER_SM)
        ++k;
    L.sub = base * k;
    L.smem = ddc_smem_bytes(T, D, L.G.wr, L.sub, &L.ring, &L.taps_pad);
    *out = L;
    return SPX_OK;
}

}  // namespace spx

using namespace spx;

struct spx_ddc : FirHandle {
    unsigned long long phase_inc = 0;
    DdcLaunch launch{};
};

namespace spx {

// K9 over samples [0, L) of `in` (device), global index of sample 0 = n0, outputs -> out (device)
static int ddc_launch(spx_ddc* d, const void* in, long long L, unsigned long long n0, float* out, cudaStream_t st) {
    const long long M = d->out_count(L);
    if (M <= 0) return SPX_OK;
    const DdcLaunch& G = d->launch;
    DdcParams p;
    p.in = in;
    p.L = L;
    p.n0 = n0;
    p.inc = d->phase_inc;
    p.taps = d->d_taps;
    p.out = out;
    p.M = M;
    p.sub = G.sub;
    p.n_sub = (M + G.sub - 1) / G.sub;
    p.scale = d->in_scale;
    p.T = d->n_taps;
    p.D = d->decim;
    p.ring = G.ring;
    p.taps_pad = G.taps_pad;
    p.s = G.G.s;
    p.c = G.G.c;
    p.wr = G.G.wr;
    p.wg = G.G.wg;
    const int per_sm = G.smem <= DDC_SMEM_TWO_PER_SM ? 2 : 1;
    const long long cap = (long long)per_sm * (d->sm_count > 0 ? d->sm_count : 148);
    const unsigned grid = (unsigned)(p.n_sub < cap ? p.n_sub : cap);
    void* args[] = {&p};
    SPX_CUDA(cudaLaunchKernel(d->kern, dim3(grid), dim3(DDC_THREADS), args, G.smem, st));
    return SPX_OK;
}

// Host memory: pieces of about piece_bytes of input (FirHandle::host_pieces); the outputs land in one device buffer and
// each piece's outputs drain on s_d2h.
static int ddc_exec_host(spx_ddc* d, const void* in, long long M, unsigned long long n0, float* out, int64_t* h2d_out,
                         int64_t* d2h_out) {
    SPX_TRY(d->st_out.reserve((size_t)M * 8));
    float* d_out = (float*)d->st_out.ptr;
    auto launch = [&](const void* d_in, long long n, long long a, long long m0, long long, int, cudaStream_t st) {
        return ddc_launch(d, d_in, n, n0 + (unsigned long long)a, d_out + 2 * m0, st);
    };
    auto drain = [&](long long m0, long long nm, int, cudaStream_t st, long long* bytes) {
        SPX_CUDA(cudaMemcpyAsync(out + 2 * m0, d_out + 2 * m0, (size_t)nm * 8, cudaMemcpyDeviceToHost, st));
        *bytes = nm * 8;
        return SPX_OK;
    };
    return d->host_pieces(in, M, d->piece_outputs(M), false, launch, drain, h2d_out, d2h_out);
}

}  // namespace spx

extern "C" {

int spx_ddc_create(spx_ddc** out, const spx_ddc_config* cfg) {
    if (!out || !cfg) return spx_set_error(SPX_E_INVALID, "NULL argument");
    *out = nullptr;
    if (cfg->struct_size != sizeof(spx_ddc_config))
        return spx_set_error(SPX_E_INVALID, "spx_ddc_config.struct_size %u != %zu", cfg->struct_size, sizeof(spx_ddc_config));
    if (cfg->decim < 1) return spx_set_error(SPX_E_INVALID, "decim %d must be >= 1", cfg->decim);
    if (cfg->n_taps < 1 || cfg->n_taps > DDC_MAX_TAPS)
        return spx_set_error(SPX_E_INVALID,
                             "n_taps %d must be in [1, %d]; for a larger decimation cascade two DDCs, the second with "
                             "shift 0", cfg->n_taps, DDC_MAX_TAPS);
    if (!cfg->taps) return spx_set_error(SPX_E_INVALID, "taps is NULL");
    if (cfg->in_fmt != SPX_FMT_CF32 && cfg->in_fmt != SPX_FMT_CI16) return spx_set_error(SPX_E_INVALID, "unknown in_fmt %d", cfg->in_fmt);
    int max_smem = 0, sms = 0;
    SPX_TRY(fir_device(cfg->device, &max_smem, &sms));
    DdcLaunch launch;
    SPX_TRY(ddc_plan_launch(cfg->n_taps, cfg->decim, max_smem, &launch));
    spx_ddc* d = new (std::nothrow) spx_ddc();
    if (!d) return spx_set_error(SPX_E_NOMEM, "out of host memory");
    d->phase_inc = (unsigned long long)cfg->phase_inc;
    d->launch = launch;
    const void* kern = cfg->in_fmt == SPX_FMT_CI16 ? (const void*)ddc_kernel<SPX_FMT_CI16> : (const void*)ddc_kernel<SPX_FMT_CF32>;
    const int rc = d->setup(*cfg, kern, max_smem, sms);
    if (rc != SPX_OK) {
        spx_ddc_destroy(d);
        return rc;
    }
    *out = d;
    return SPX_OK;
}

int spx_ddc_destroy(spx_ddc* d) {
    if (!d) return SPX_OK;
    d->release();
    delete d;
    return SPX_OK;
}

int spx_ddc_sync(spx_ddc* d) {
    if (!d) return spx_set_error(SPX_E_INVALID, "ddc is NULL");
    return d->sync();
}

int spx_ddc_exec(spx_ddc* d, int32_t mem, const void* in, int64_t n_samples, int64_t first_sample, float* out,
                 int64_t* n_out, int64_t* h2d_bytes_out, int64_t* d2h_bytes_out, void* stream) {
    if (!d) return spx_set_error(SPX_E_INVALID, "ddc is NULL");
    long long M = 0;
    std::unique_lock<std::mutex> lock;
    SPX_TRY(d->exec_begin(mem, in, n_samples, first_sample, out, 4, &M, n_out, h2d_bytes_out, d2h_bytes_out, &lock));
    if (M == 0) return SPX_OK;
    if (mem == SPX_MEM_DEVICE)
        return ddc_launch(d, in, n_samples, (unsigned long long)first_sample, out, stream ? (cudaStream_t)stream : d->s_compute);
    return ddc_exec_host(d, in, M, (unsigned long long)first_sample, out, h2d_bytes_out, d2h_bytes_out);
}

}  // extern "C"
