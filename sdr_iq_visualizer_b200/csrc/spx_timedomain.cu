// spx_timedomain.cu -- K4: time-domain / constellation views.
//
//   * per-frame mean and peak power  mean(I^2+Q^2), max(I^2+Q^2)  (SURVEY.md 8(a) A9; the reference
//     only prints 20*log10(mean|x|) per buffer, /root/reference/scripts/pyad-iio-test.py:93)
//   * 2-D I/Q density histogram with np.histogram2d semantics (A10) replacing the random 2000-point
//     constellation scatter of /root/reference/app/dashboard/callbacks.py:199-214.  Counts are
//     integers and must be bit-exact: the bin of a value is decided against the float64 edge
//     table exactly as numpy builds it (linspace: fl(fl(i*step) + start), last edge = stop).
#include <math.h>
#include <string.h>

#include <mutex>

#include "spx_internal.h"
#include "spx_plan.h"

namespace spx {

struct HistGrid {
    double start, stop, step, inv_step;
    int bins;
};

// Per-launch constants of the shared-memory histogram kernel, built on the host (as kernel parameters they are constant-bank
// operands; derived inside the kernel the compiler rebuilds them per sample to save registers).
struct HistConst {
    float fa, fb;         // bin estimate u = fa * x + fb = (x * scale - start) / step - 1/2
    float neg_center;     // -(bins - 1) / 2
    float half_bins;      // bins / 2
    float zone;           // |u - rint(u)| at or above this: within HIST_EPS of an edge, settled exactly (2: never, see hist_constants)
    int idx_bias;         // 0x4B400000 * (bins + 1)
    int swz_mask;         // 31 when every table row starts on a 32-word boundary (bins % 64 == 0), else 0
};

__device__ __forceinline__ double edge_of(const HistGrid& g, int i) {
    return i >= g.bins ? g.stop : __dadd_rn(__dmul_rn((double)i, g.step), g.start);
}

// np.searchsorted(edges, v, 'right') - 1 with the right edge closed; -1 = outside.
// Branch-light and exact: the float64 estimate floor((v - start) / step) is at most one bin off, so one comparison
// against the lower edge and one against the upper edge -- both built exactly as numpy builds them -- settle it.
__device__ __forceinline__ int bin_of(const HistGrid& g, double v) {
    const double t = (v - g.start) * g.inv_step;
    int b = __double2int_rd(t);
    b = max(0, min(b, g.bins - 1));
    const double e0 = edge_of(g, b);
    b -= (v < e0) ? 1 : 0;
    b = max(b, 0);
    const double e1 = edge_of(g, b + 1);
    b += (v >= e1 && b < g.bins - 1) ? 1 : 0;
    return (v >= g.start && v <= g.stop) ? b : -1;   // NaN fails both comparisons
}

template <int FMT>
__device__ __forceinline__ void load_iq(const void* in, long long i, double scale, double& re, double& im) {
    if (FMT == SPX_FMT_CF32) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(in) + i);
        re = (double)v.x * scale;
        im = (double)v.y * scale;
    } else {
        const short2 v = __ldg(reinterpret_cast<const short2*>(in) + i);
        re = (double)v.x * scale;
        im = (double)v.y * scale;
    }
}

__device__ __forceinline__ void hist_count(const HistGrid& g, unsigned int* hist, double re, double im) {
    const int bi = bin_of(g, re), bq = bin_of(g, im);
    if (bi >= 0 && bq >= 0) atomicAdd(hist + (size_t)bi * g.bins + bq, 1u);  // H[i][j], i <-> I, j <-> Q
}

// Streaming pass over the samples: every thread issues four independent 16-byte loads (2 cf32 or 4 ci16 samples each,
// ld.global.nc, no L1 allocation) before it touches any of them, so 64 bytes per thread are in flight and the pass is
// bandwidth- rather than latency-bound on cold input; the counts go to the L2-resident table with RED.ADD.
// (`vec_ok` = the buffer is 16-byte aligned; otherwise, and for the tail, samples are read one at a time.)
template <int FMT>
__global__ void __launch_bounds__(256) hist2d_kernel(const void* __restrict__ in, long long n, double scale, HistGrid g,
                                                     unsigned int* __restrict__ hist, int vec_ok) {
    constexpr int SPV = FMT == SPX_FMT_CF32 ? 2 : 4;   // samples per 16-byte vector
    constexpr int U = 4;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long tid0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long nvec = vec_ok ? n / SPV : 0;
    const uint4* vin = reinterpret_cast<const uint4*>(in);
    for (long long v0 = tid0; v0 < nvec; v0 += stride * U) {
        uint4 w[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const long long vi = v0 + u * stride;
            w[u] = make_uint4(0u, 0u, 0u, 0u);
            if (vi < nvec)
                asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(w[u].x), "=r"(w[u].y), "=r"(w[u].z), "=r"(w[u].w) : "l"(vin + vi));
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (v0 + u * stride >= nvec) break;
            const unsigned int q[4] = {w[u].x, w[u].y, w[u].z, w[u].w};
            if (FMT == SPX_FMT_CF32) {
                hist_count(g, hist, (double)__uint_as_float(q[0]) * scale, (double)__uint_as_float(q[1]) * scale);
                hist_count(g, hist, (double)__uint_as_float(q[2]) * scale, (double)__uint_as_float(q[3]) * scale);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    hist_count(g, hist, (double)(short)(q[k] & 0xffffu) * scale, (double)(short)(q[k] >> 16) * scale);
            }
        }
    }
    for (long long i = nvec * SPV + tid0; i < n; i += stride) {   // tail (or everything, when unaligned)
        double re, im;
        load_iq<FMT>(in, i, scale, re, im);
        hist_count(g, hist, re, im);
    }
}

// Shared-memory privatised variant (north_star: "a shared-memory I/Q 2-D histogram for the constellation view"), used
// when bins^2 16-bit counters fit in 200 KB of shared memory (bins <= 318; 128 KB for 256 x 256).  Real constellations pile up
// on a few thousand bins, and RED.ADD on the same L2 sectors from every SM serialises (ncu: 261 us for 2^24 samples with
// the global-atomic kernel above, DRAM at 6 %).  Here every CTA keeps ONE table of packed 16-bit counters in shared memory
// for its whole share of the input (two per word, ATOMS.ADD of 1 or 1<<16):
//   * the input is walked in epochs of <= 57 344 samples; between two epochs the CTA scans its table and moves every
//     counter that has reached 2^13 to the global table (RED, rare), so a counter starts an epoch below 2^13 and cannot wrap;
//   * at the end the table is written as it is (packed, coalesced stores) to the CTA's private slice of `tabs`, and
//     hist_merge_kernel adds the slices up -- no atomics on the way out.  Round 2 measured why: flushing each 65 528-sample
//     chunk with RED put ~5 M atomics on one L2-resident table (92-141 G/s, tools/micro/atom_mix.cu), 50 of the 58 us;
//     the shared-memory atomics themselves run at 2.5-4.8 per clock and SM (12-23 us for 2^24 samples).
//   * `tabs == nullptr` (a handful of CTAs): non-zero counters go straight to the global table with RED.
// Neighbouring floats (finite, non-NaN arguments).
__device__ __forceinline__ float float_up(float x) {
    if (x == 0.f) return __int_as_float(1);
    const int b = __float_as_int(x);
    return __int_as_float(x > 0.f ? b + 1 : b - 1);
}
__device__ __forceinline__ float float_down(float x) { return -float_up(-x); }

template <int FMT>
__global__ void __launch_bounds__(1024) hist2d_smem_kernel(const void* __restrict__ in, long long n, double scale, HistGrid g,
                                                           unsigned int* __restrict__ hist, int vec_ok, long long span,
                                                           unsigned int* __restrict__ tabs, int tab_stride, HistConst hc) {
    extern __shared__ __align__(16) unsigned int sh[];
    constexpr int SPV = FMT == SPX_FMT_CF32 ? 2 : 4;   // samples per 16-byte vector
    constexpr int U = FMT == SPX_FMT_CF32 ? 4 : 2;     // vectors per thread and batch: 8 samples, 8192 per CTA
    constexpr int STEP = 1024 * U;                     // vectors per CTA and batch (the launch uses 1024 threads)
    constexpr int EPOCH_BATCHES = 7;                   // 57 344 samples between two scans for hot counters: 8191 + 57 344 = 65 535
    constexpr int EPOCH_SCALAR = 57344;
    constexpr unsigned HOT = 0xE000E000u;              // a counter >= 2^13 (either half of a word)
    const int tid = threadIdx.x;
    const int bins = g.bins, nb2 = bins * bins, words = (nb2 + 1) / 2, quads = (words + 3) / 4;
    uint4* sh4 = reinterpret_cast<uint4*>(sh);
    // Programmatic dependent launch: the merge kernel behind this one may be scheduled now (it waits for this grid to
    // complete before it reads); this grid's prologue (zeroed table, thresholds) overlaps the tail of what is in front of it.
    asm volatile("griddepcontrol.launch_dependents;");
    // The exact decision, in the units of the raw input: thr[i] = the smallest float x whose value v = (double)x * scale
    // reaches numpy's edge i (v >= e_i  <=>  x >= thr[i], the product is monotone in x for scale > 0), thr[bins + 1] = the
    // largest x with v <= stop.  Built once per CTA from the float64 edges; comparing a sample against two neighbouring
    // thresholds settles its bin exactly, in float, with two shared-memory loads.
    float* thr = reinterpret_cast<float*>(sh + 4 * quads);
    for (int i = tid; i <= bins + 1; i += 1024) {
        const double e = i <= bins ? edge_of(g, i) : g.stop;
        float x = (float)(e / scale);
        if (i <= bins) {
            while ((double)x * scale >= e && x > -3.0e38f) x = float_down(x);
            while ((double)x * scale < e && x < 3.0e38f) x = float_up(x);
        } else {
            while ((double)x * scale <= e && x < 3.0e38f) x = float_up(x);
            while ((double)x * scale > e && x > -3.0e38f) x = float_down(x);
        }
        thr[i] = x;
    }
    for (int q = tid; q < quads; q += 1024) sh4[q] = make_uint4(0u, 0u, 0u, 0u);
    // the swizzle needs every row to start on a 32-word boundary (bins a multiple of 64); otherwise it is switched off
    const int swz_mask = hc.swz_mask;
    // Bin estimate u = (v - start)/step - 1/2 as ONE fma in float (constants rounded from float64): its error is below
    // 4e-5 bins for bins <= 320 (|u| <= 160: half an ulp of the product, of the constant and of the result, 1.5e-5 each
    // at most).  rint(u) through the 1.5 * 2^23 constant: when u is farther than HIST_EPS = 2e-4 from a half-integer, i.e.
    // (v - start)/step is farther than HIST_EPS from an edge, and inside the range, rint(u) IS the bin; otherwise the
    // threshold table decides (and drops what is outside [start, stop], infinite or NaN, as numpy does).
    // I and Q go through the four arithmetic steps as one packed pair (FFMA2 / FADD2).
    constexpr float MAGIC = 12582912.0f;
    constexpr int MAGIC_BITS = 0x4B400000;
    const float2 fa2 = make_float2(hc.fa, hc.fa), fb2 = make_float2(hc.fb, hc.fb), mg2 = make_float2(MAGIC, MAGIC), nmg2 = make_float2(-MAGIC, -MAGIC),
                 neg2 = make_float2(-1.f, -1.f);
    unsigned sh_base = (unsigned)__cvta_generic_to_shared(sh);
    asm volatile("" : "+r"(sh_base));   // keep the base in a register (otherwise it is rebuilt from SR_CgaCtaId per sample)
    // range test on the estimate itself: rint(u) in [0, bins) <=> |u - (bins - 1)/2| < bins/2 away from the two outer edges
    // (both constants exact in float; at the outer edges the exact path decides)
    const float2 nctr2 = make_float2(hc.neg_center, hc.neg_center);
    const float half_bins = hc.half_bins;
    const int idx_bias = hc.idx_bias;   // (bits(m.x) * bins + bits(m.y)) - idx_bias = bi * bins + bq  (mod 2^32)
    // exact bin of raw component x (or -1: outside [start, stop], NaN); `est` is at most one bin off for values in range and
    // arbitrary (clamped) for far outliers, which fail the range test
    auto settle = [&](float x, int est) -> int {
        int b = max(0, min(est, bins - 1));
        b -= (x < thr[b]) ? 1 : 0;
        b = max(b, 0);
        b += (x >= thr[b + 1] && b < bins - 1) ? 1 : 0;
        return (x >= thr[0] && x <= thr[bins + 1]) ? b : -1;
    };
    const float zone = hc.zone;
    auto count_f = [&](float2 f) {
        const float2 u = __ffma2_rn(f, fa2, fb2);
        const float2 m = __fadd2_rn(u, mg2);
        const float2 d = __ffma2_rn(__fadd2_rn(m, nmg2), neg2, u);            // u - rint(u), exact, in [-0.5, 0.5]
        const float2 c = __fadd2_rn(u, nctr2);
        int idx = __float_as_int(m.x) * bins + __float_as_int(m.y) - idx_bias;
        int swz = __float_as_int(m.x) & swz_mask;                              // = bi & swz_mask: the low bits of MAGIC_BITS are 0
        // the estimate is the answer when both components are clear of every edge and inside the range (two compares for
        // the range, not fmaxf: a NaN must fail); everything else is settled exactly, or dropped
        if (!(fabsf(c.x) < half_bins && fabsf(c.y) < half_bins) || fmaxf(fabsf(d.x), fabsf(d.y)) >= zone) {
            const int bi = settle(f.x, __float_as_int(m.x) - MAGIC_BITS), bq = settle(f.y, __float_as_int(m.y) - MAGIC_BITS);
            if ((bi | bq) < 0) return;
            idx = bi * bins + bq;
            swz = bi & swz_mask;
        }
        // Bank swizzle.  With idx = bi * bins + bq the bank of a counter depends on bq alone (bins/2 words per row is a
        // multiple of 32 for 256 bins), and a constellation cluster is ~15 bins wide: the 32 lanes of a warp fell on ~8
        // banks (ncu: 46.8 % of the shared wavefronts were conflicts).  XOR-ing the word index with the row number spreads
        // a cluster over all banks; it is a bijection inside each aligned group of 32 words, undone by hist_merge_kernel.
        // (Integer multiply-adds instead of shifts / selects: the FMA pipe has twice the ALU pipe's rate.)
        unsigned int val, addr;
        asm volatile("mad.lo.u32 %0, %1, 65535, 1;" : "=r"(val) : "r"((unsigned)idx & 1u));
        asm volatile("mad.lo.u32 %0, %1, 4, %2;" : "=r"(addr) : "r"((unsigned)((idx >> 1) ^ swz)), "r"(sh_base));
        asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(val) : "memory");
    };
    auto count_vec = [&](const uint4& wv) {
        if (FMT == SPX_FMT_CF32) {
            count_f(make_float2(__uint_as_float(wv.x), __uint_as_float(wv.y)));
            count_f(make_float2(__uint_as_float(wv.z), __uint_as_float(wv.w)));
        } else {
            const unsigned int q[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) count_f(make_float2((float)(short)(q[k] & 0xffffu), (float)(short)(q[k] >> 16)));
        }
    };
    auto unswizzled = [&](int w) { return swz_mask ? (w ^ ((2 * w / bins) & swz_mask)) : w; };   // row = 2 w / bins
    // Between two epochs: every counter that has reached 2^13 moves to the global table, so no counter can wrap in the
    // next epoch (< 2^13 at its start, <= 57 344 increments).  All threads of the CTA call this.
    auto move_hot_counters = [&]() {
        __syncthreads();
        for (int q = tid; q < quads; q += 1024) {
            const uint4 v4 = sh4[q];
            if (((v4.x | v4.y | v4.z | v4.w) & HOT) == 0u) continue;
            const unsigned int vv[4] = {v4.x, v4.y, v4.z, v4.w};
            for (int k = 0; k < 4; ++k) {
                const unsigned int v = vv[k];
                if ((v & HOT) == 0u) continue;
                const int wo = unswizzled(4 * q + k);
                unsigned int keep = v;
                if (v & (HOT & 0xffffu)) { atomicAdd(hist + 2 * wo, v & 0xffffu); keep &= 0xffff0000u; }
                if (v & (HOT & 0xffff0000u)) { atomicAdd(hist + 2 * wo + 1, v >> 16); keep &= 0x0000ffffu; }
                sh[4 * q + k] = keep;
            }
        }
        __syncthreads();
    };
    asm volatile("griddepcontrol.wait;" ::: "memory");   // the input and the zeroed histogram are complete and visible from here
    __syncthreads();
    // this CTA's share of the input: [s0, s1), s0 a multiple of 8 samples
    const long long s0 = (long long)blockIdx.x * span, s1 = (s0 + span < n) ? s0 + span : n;
    long long done = s0;
    if (vec_ok && s0 < s1) {
        // Software pipeline over batches of U vectors per thread: the loads of batch k + 1 are in flight while batch k is
        // counted (and while the hot-counter scan runs), ld.global.nc without L1 allocation.
        const long long v_lo = s0 / SPV, v_hi = s1 / SPV;
        const uint4* p = reinterpret_cast<const uint4*>(in) + v_lo + tid;
        long long rem = v_hi - v_lo;   // vectors of this share from the current batch on (uniform)
        uint4 cur[U], nxt[U];
        auto fetch = [&](uint4* dst, const uint4* q, long long left) {
            const int lim = left < (long long)STEP ? (int)(left > 0 ? left : 0) : STEP;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                dst[u] = make_uint4(0u, 0u, 0u, 0u);
                if (tid + 1024 * u < lim)
                    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(dst[u].x), "=r"(dst[u].y), "=r"(dst[u].z), "=r"(dst[u].w) : "l"(q + 1024 * u));
            }
        };
        fetch(cur, p, rem);
        int batches = 0;
#pragma unroll 1
        while (rem > 0) {
            fetch(nxt, p + STEP, rem - STEP);
            if (rem >= STEP) {   // full batch (uniform per CTA): no per-vector bounds
#pragma unroll
                for (int u = 0; u < U; ++u) count_vec(cur[u]);
            } else {
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (tid + 1024 * u < (int)rem) count_vec(cur[u]);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) cur[u] = nxt[u];
            p += STEP;
            rem -= STEP;
            if (++batches == EPOCH_BATCHES && rem > 0) {
                move_hot_counters();
                batches = 0;
            }
        }
        done = v_hi * SPV;
    }
    // tail, or the whole share when the buffer is not 16-byte aligned: one sample at a time, epochs of 57 344
    for (long long e0 = done; e0 < s1; e0 += EPOCH_SCALAR) {
        const long long e1 = (e0 + EPOCH_SCALAR < s1) ? e0 + EPOCH_SCALAR : s1;
        if (e0 != s0) move_hot_counters();
        for (long long i = e0 + tid; i < e1; i += 1024) {
            if (FMT == SPX_FMT_CF32) {
                count_f(__ldg(reinterpret_cast<const float2*>(in) + i));
            } else {
                const short2 v = __ldg(reinterpret_cast<const short2*>(in) + i);
                count_f(make_float2((float)v.x, (float)v.y));
            }
        }
    }
    __syncthreads();
    if (tabs != nullptr) {   // the table as it is (swizzled, packed); tab_stride is a multiple of 4 words
        uint4* my = reinterpret_cast<uint4*>(tabs + (size_t)blockIdx.x * tab_stride);
        for (int q = tid; q < quads; q += 1024) my[q] = sh4[q];
    } else {
        for (int w = tid; w < words; w += 1024) {
            const unsigned int v = sh[w];
            const int wo = unswizzled(w);
            if (v & 0xffffu) atomicAdd(hist + 2 * wo, v & 0xffffu);
            if (v >> 16) atomicAdd(hist + 2 * wo + 1, v >> 16);
        }
    }
}

// Sum of the CTA-private packed tables into the uint32 histogram: thread (w, q) adds tables q, q + 4, ... for word w
// (read at its swizzled position), the four partial sums meet in shared memory.  Reads ntabs x 128 KB from L2, plain
// read-modify-write of `hist` (stream-ordered behind the counting kernel, nothing else touches it).
__global__ void __launch_bounds__(256) hist_merge_kernel(const unsigned int* __restrict__ tabs, int ntabs, int tab_stride, int words,
                                                         int bins, unsigned int* __restrict__ hist) {
    __shared__ unsigned int part[2][4][64];
    asm volatile("griddepcontrol.wait;" ::: "memory");   // launched early (programmatic dependent launch): wait for the tables
    const int wl = threadIdx.x & 63, q = threadIdx.x >> 6, w = blockIdx.x * 64 + wl;
    const int swz_mask = (bins % 64 == 0) ? 31 : 0;
    unsigned int lo = 0u, hi = 0u;
    if (w < words) {
        const int ws = swz_mask ? (w ^ ((2 * w / bins) & swz_mask)) : w;
#pragma unroll 8
        for (int t = q; t < ntabs; t += 4) {
            const unsigned int v = __ldcg(tabs + (size_t)t * tab_stride + ws);
            lo += v & 0xffffu;
            hi += v >> 16;
        }
    }
    part[0][q][wl] = lo;
    part[1][q][wl] = hi;
    __syncthreads();
    if (threadIdx.x < 128) {
        const int h = threadIdx.x >> 6, bin = 2 * w + h;
        const unsigned int sum = part[h][0][wl] + part[h][1][wl] + part[h][2][wl] + part[h][3][wl];
        if (w < words && bin < bins * bins && sum) hist[bin] += sum;
    }
}

// Zeroes the histogram in front of the counting kernel (instead of a memset node, so that the counting kernel can be a
// programmatic dependent launch and run its prologue next to this).
__global__ void __launch_bounds__(256) hist_zero_kernel(unsigned int* __restrict__ hist, int n) {
    asm volatile("griddepcontrol.launch_dependents;");
    for (int i = blockIdx.x * 256 + threadIdx.x; i < n; i += gridDim.x * 256) hist[i] = 0u;
}

template <int FMT>
__global__ void __launch_bounds__(256) frame_stats_kernel(const void* __restrict__ in, long long n_frames, int frame_len,
                                                          int hop, float scale, float* __restrict__ mean_pow,
                                                          float* __restrict__ peak_pow) {
    __shared__ double s_sum[8];
    __shared__ float s_max[8];
    for (long long f = blockIdx.x; f < n_frames; f += gridDim.x) {
        const long long base = f * hop;
        double sum = 0.0;
        float mx = 0.f;
        for (int j = threadIdx.x; j < frame_len; j += 256) {
            float re, im;
            if (FMT == SPX_FMT_CF32) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(in) + base + j);
                re = v.x * scale; im = v.y * scale;
            } else {
                const short2 v = __ldg(reinterpret_cast<const short2*>(in) + base + j);
                re = (float)v.x * scale; im = (float)v.y * scale;
            }
            const float p = re * re + im * im;
            sum += (double)p;
            mx = fmaxf(mx, p);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sum += __shfl_xor_sync(0xffffffffu, sum, o);
            mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        __syncthreads();
        if ((threadIdx.x & 31) == 0) { s_sum[threadIdx.x >> 5] = sum; s_max[threadIdx.x >> 5] = mx; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            float m = 0.f;
            for (int w = 0; w < 8; ++w) { t += s_sum[w]; m = fmaxf(m, s_max[w]); }
            mean_pow[f] = (float)(t / (double)frame_len);
            peak_pow[f] = m;
        }
    }
}

// Constants of the bin estimate.  General case: u = (x * scale - start)/step - 1/2 with an edge zone of HIST_EPS bins.
// Integer input on a power-of-two grid (ci16, scale = 2^a, step = 2^b, e.g. R = 2048 / 256 bins, or the SigMF scale 2^-15
// with R = 1): every product, sum and numpy edge is exact, t = (v - start)/step is a multiple of G = min(2^(a-b), 1) and a
// sixteenth of such samples sits exactly ON an edge.  Shifting the estimate by G/2 makes rint(t - 1/2 + G/2) = floor(t)
// for every sample, ties included, so the edge zone is switched off; only v = stop (t = bins) and values outside the range
// fail the range test and take the threshold table.
static HistConst hist_constants(const HistGrid& g, int in_fmt, double scale) {
    HistConst hc;
    const int bins = g.bins;
    double shift = 0.0;
    hc.zone = 0.5f - 2e-4f;
    if (in_fmt == SPX_FMT_CI16) {
        int ea = 0, eb = 0;
        const double ma = frexp(scale, &ea), mb = frexp(g.step, &eb);
        const int k = ea - eb;   // scale / step = 2^k when both mantissas are 1/2
        const bool exact_edges = g.step * bins == g.stop - g.start && g.start == -g.stop;
        if (ma == 0.5 && mb == 0.5 && exact_edges && k >= -11 && k <= 6) {
            shift = k < 0 ? ldexp(1.0, k - 1) : 0.25;
            hc.zone = 2.0f;
        }
    }
    hc.fa = (float)(scale * g.inv_step);
    hc.fb = (float)(-g.start * g.inv_step - 0.5 + shift);
    hc.neg_center = -0.5f * (float)(bins - 1);
    hc.half_bins = 0.5f * (float)bins;
    hc.idx_bias = (int)(0x4B400000u * (unsigned)(bins + 1));
    hc.swz_mask = (bins % 64 == 0) ? 31 : 0;
    return hc;
}

}  // namespace spx

using namespace spx;

extern "C" int spx_iq_hist2d(int32_t device, int32_t mem, const void* in, int32_t in_fmt, double in_scale, int64_t n,
                             double r, int32_t bins, uint32_t* hist, int32_t accumulate, void* stream) {
    if (!hist) return spx_set_error(SPX_E_INVALID, "hist is NULL");
    if (bins < 1 || bins > 4096 || !(r > 0.0)) return spx_set_error(SPX_E_INVALID, "need 1 <= bins <= 4096 and R > 0");
    if (in_fmt != SPX_FMT_CF32 && in_fmt != SPX_FMT_CI16) return spx_set_error(SPX_E_INVALID, "unknown in_fmt");
    if (n < 0 || (n > 0 && !in)) return spx_set_error(SPX_E_INVALID, "bad input");
    DeviceCtx* ctx;
    SPX_TRY(device_ctx(device, &ctx));
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaStream_t st = (mem == SPX_MEM_DEVICE && stream) ? (cudaStream_t)stream : ctx->st;
    HistGrid g;
    g.start = -r;
    g.stop = r;
    g.step = (g.stop - g.start) / (double)bins;  // numpy linspace: delta / div
    g.inv_step = 1.0 / g.step;
    g.bins = bins;
    const size_t esz = in_fmt == SPX_FMT_CI16 ? 4 : 8, hbytes = (size_t)bins * bins * sizeof(uint32_t);
    const void* d_in = in;
    unsigned int* d_hist = hist;
    if (mem == SPX_MEM_HOST) {
        void* part[2];
        SPX_TRY(ctx->carve({(size_t)n * esz, hbytes}, part));
        if (n) SPX_CUDA(cudaMemcpyAsync(part[0], in, (size_t)n * esz, cudaMemcpyHostToDevice, st));
        d_in = part[0];
        d_hist = (unsigned int*)part[1];
        if (accumulate) SPX_CUDA(cudaMemcpyAsync(d_hist, hist, hbytes, cudaMemcpyHostToDevice, st));
    }
    bool zeroed = accumulate != 0;
    if (n > 0) {
        const int sm = ctx->sm_count;
        const int vec_ok = ((uintptr_t)d_in & 15u) == 0 ? 1 : 0;
        const size_t words = (size_t)((bins * bins + 1) / 2);
        const size_t smem = ((words + 3) & ~(size_t)3) * sizeof(unsigned int) + (size_t)(bins + 2) * sizeof(float);
        if (smem <= 200u * 1024u && in_scale > 0.0 && in_scale < 1e30) {
            // shared-memory privatised counting: one CTA per SM, each with a contiguous share of the input (a multiple of 8
            // samples, at least one epoch so that small inputs do not spread over CTAs that each dump a table)
            auto kern = in_fmt == SPX_FMT_CF32 ? hist2d_smem_kernel<SPX_FMT_CF32> : hist2d_smem_kernel<SPX_FMT_CI16>;
            SPX_TRY(kernel_setup((const void*)kern, 1024, 200 * 1024, nullptr));
            long long span = ((n + sm - 1) / sm + 7) & ~7ll;
            if (span < 32760) span = 32760;
            const long long blocks = (n + span - 1) / span;
            const HistConst hc = hist_constants(g, in_fmt, in_scale);
            unsigned int* tabs = nullptr;
            const int tab_stride = (int)((words + 3) & ~(size_t)3);
            if (blocks > 4) {
                if (!ctx->hist_pool) {
                    cudaMemPoolProps props;
                    memset(&props, 0, sizeof(props));
                    props.allocType = cudaMemAllocationTypePinned;
                    props.location.type = cudaMemLocationTypeDevice;
                    props.location.id = device;
                    SPX_CUDA(cudaMemPoolCreate(&ctx->hist_pool, &props));
                    unsigned long long keep = ~0ull;   // freed blocks stay in the pool: the next call reuses them
                    SPX_CUDA(cudaMemPoolSetAttribute(ctx->hist_pool, cudaMemPoolAttrReleaseThreshold, &keep));
                }
                SPX_CUDA(cudaMallocFromPoolAsync((void**)&tabs, (size_t)blocks * tab_stride * sizeof(unsigned int), ctx->hist_pool, st));
            }
            cudaLaunchAttribute pdl[1];
            pdl[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            pdl[0].val.programmaticStreamSerializationAllowed = 1;
            cudaLaunchConfig_t cfg = {};
            cfg.stream = st;
            cfg.attrs = pdl;
            cfg.numAttrs = 1;
            if (!zeroed) {
                hist_zero_kernel<<<64, 256, 0, st>>>(d_hist, bins * bins);
                zeroed = true;
            }
            cfg.gridDim = dim3((unsigned)blocks);
            cfg.blockDim = dim3(1024);
            cfg.dynamicSmemBytes = smem;
            SPX_CUDA(cudaLaunchKernelEx(&cfg, kern, d_in, (long long)n, in_scale, g, d_hist, vec_ok, span, tabs, tab_stride, hc));
            if (tabs) {
                cfg.gridDim = dim3((unsigned)((words + 63) / 64));
                cfg.blockDim = dim3(256);
                cfg.dynamicSmemBytes = 0;
                SPX_CUDA(cudaLaunchKernelEx(&cfg, hist_merge_kernel, (const unsigned int*)tabs, (int)blocks, tab_stride, (int)words, bins, d_hist));
                SPX_CUDA(cudaFreeAsync(tabs, st));
            }
        } else {
            if (!zeroed) {
                SPX_CUDA(cudaMemsetAsync(d_hist, 0, hbytes, st));
                zeroed = true;
            }
            long long blocks = (n + 255) / 256;
            if (blocks > (long long)sm * 8) blocks = (long long)sm * 8;
            if (in_fmt == SPX_FMT_CF32) hist2d_kernel<SPX_FMT_CF32><<<(unsigned)blocks, 256, 0, st>>>(d_in, n, in_scale, g, d_hist, vec_ok);
            else hist2d_kernel<SPX_FMT_CI16><<<(unsigned)blocks, 256, 0, st>>>(d_in, n, in_scale, g, d_hist, vec_ok);
        }
        SPX_CUDA(cudaGetLastError());
    }
    if (!zeroed) SPX_CUDA(cudaMemsetAsync(d_hist, 0, hbytes, st));   // n == 0
    if (mem == SPX_MEM_HOST) {
        SPX_CUDA(cudaMemcpyAsync(hist, d_hist, hbytes, cudaMemcpyDeviceToHost, st));
        SPX_CUDA(cudaStreamSynchronize(st));
    }
    return SPX_OK;
}

extern "C" int spx_frame_stats(int32_t device, int32_t mem, const void* in, int32_t in_fmt, float in_scale, int64_t n,
                               int32_t frame_len, int32_t hop, float* mean_pow, float* peak_pow, int64_t* n_frames_out,
                               void* stream) {
    if (frame_len < 1 || hop < 1) return spx_set_error(SPX_E_INVALID, "frame_len and hop must be >= 1");
    if (in_fmt != SPX_FMT_CF32 && in_fmt != SPX_FMT_CI16) return spx_set_error(SPX_E_INVALID, "unknown in_fmt");
    const long long F = n < frame_len ? 0 : (n - frame_len) / hop + 1;
    if (n_frames_out) *n_frames_out = F;
    if (F == 0) return SPX_OK;
    if (!in || !mean_pow || !peak_pow) return spx_set_error(SPX_E_INVALID, "NULL buffer");
    DeviceCtx* ctx;
    SPX_TRY(device_ctx(device, &ctx));
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaStream_t st = (mem == SPX_MEM_DEVICE && stream) ? (cudaStream_t)stream : ctx->st;
    const size_t esz = in_fmt == SPX_FMT_CI16 ? 4 : 8;
    const void* d_in = in;
    float *d_mean = mean_pow, *d_peak = peak_pow;
    if (mem == SPX_MEM_HOST) {
        void* part[2];
        SPX_TRY(ctx->carve({(size_t)n * esz, (size_t)F * 2 * sizeof(float)}, part));
        SPX_CUDA(cudaMemcpyAsync(part[0], in, (size_t)n * esz, cudaMemcpyHostToDevice, st));
        d_in = part[0];
        d_mean = (float*)part[1];
        d_peak = d_mean + F;
    }
    const int sm = ctx->sm_count;
    long long blocks = F < (long long)sm * 8 ? F : (long long)sm * 8;
    if (in_fmt == SPX_FMT_CF32)
        frame_stats_kernel<SPX_FMT_CF32><<<(unsigned)blocks, 256, 0, st>>>(d_in, F, frame_len, hop, in_scale, d_mean, d_peak);
    else
        frame_stats_kernel<SPX_FMT_CI16><<<(unsigned)blocks, 256, 0, st>>>(d_in, F, frame_len, hop, in_scale, d_mean, d_peak);
    SPX_CUDA(cudaGetLastError());
    if (mem == SPX_MEM_HOST) {
        SPX_CUDA(cudaMemcpyAsync(mean_pow, d_mean, (size_t)F * sizeof(float), cudaMemcpyDeviceToHost, st));
        SPX_CUDA(cudaMemcpyAsync(peak_pow, d_peak, (size_t)F * sizeof(float), cudaMemcpyDeviceToHost, st));
        SPX_CUDA(cudaStreamSynchronize(st));
    }
    return SPX_OK;
}
