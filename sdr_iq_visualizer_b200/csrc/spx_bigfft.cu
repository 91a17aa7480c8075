// spx_bigfft.cu -- K2: STFT for N = N1*N2 in [16384, 1048576] (BASELINE config 5: N = 65536).
//
// A 65536-point frame is 512 KiB of cf32 and cannot live in one CTA's shared memory, so the
// transform is split four-step style into two fused kernels that meet in an L2-resident scratch
// (frames are processed in batches sized to the 126 MB L2):
//
//   A (columns): for G adjacent columns n2 of the [N1][N2] view of a frame, load
//       x[N2*n1 + n2] * w[N2*n1 + n2] (unpack + window fused; 128-byte row segments), do the N1-point
//       Stockham FFT over n1 in shared memory, multiply by W_N^{n2*k1} (two-level table) and store
//       T[k1][n2] (coalesced along n2).
//   B (rows): for FPC adjacent rows k1 of T, do the N2-point FFT over n2; bin k = k1 + N1*k2.  The
//       fused epilogue (|X|^2, dB, fftshift, Welch, max-hold, u8) is the same as K1's; the dB / u8
//       values are transposed through shared memory so that global stores are runs of FPC bins.
//
// Replaces np.fft.fft for long frames (/root/reference/app/sdr/streamer.py:119; the 2^16-sample
// buffers of /root/reference/scripts/pyad-iio-test.py:50-61).
#include <math.h>
#include <string.h>

#include <vector>

#include "spx_plan.h"
#include "spx_async.cuh"
#include "spx_stft_device.cuh"
#include "spx_tables.h"

namespace spx {

struct BigParams {
    const void* in;          // samples of the stream (cf32 / ci16)
    long long sample0;       // first sample of the first frame of this batch
    int hop;
    int frames;              // frames in this batch
    const float* win;        // [N] window * scale or nullptr
    const float2* tw1;       // twiddles of the N1-point FFT
    const float2* tw2;       // twiddles of the N2-point FFT
    const float2* wn_fine;   // W_N^i, i in [0,256)
    const float2* wn_coarse; // W_N^(256 i), i in [0, N/256)
    float2* scratch;         // T: [frames][N1][N2]
    // outputs (rows are indexed from row0)
    long long row0;
    float* db_rows;
    unsigned char* wf_rows;
    float2* spec_rows;
    double* welch_acc;       // [N] of this stream
    float* maxhold;
    float db_eps, db_pw_min, q_a, q_b;
    int frames_per_chunk;    // kernel B: accumulator flush granularity
    int sys_atomics;         // accumulators may live on a peer GPU
};

template <int N1, int N2>
struct BigCfg {
    static constexpr int N = N1 * N2;
    // kernel A
    static constexpr int T1 = N1 / 16;
#ifndef SPX_K2_G
#define SPX_K2_G 16
#endif
#ifndef SPX_K2_THREADS_B
#define SPX_K2_THREADS_B 128   // 128-thread row CTAs: twice as many independent barrier groups per SM (+2 % on the config-5 shape)
#endif
    static constexpr int G = N1 >= 1024 ? 8 : SPX_K2_G;        // columns per CTA
    static constexpr int THREADS_A = G * T1;
    static constexpr int P1 = plan_passes(N1);
    static constexpr int BUF1 = padded_size(N1) + (P1 >= 3 ? N1 : 0);
    static constexpr int S1 = BUF1 | 1;                        // odd column stride: conflict-free across columns
    static constexpr int TW1 = plan_tw_size(N1);
    // kernel B
    static constexpr int T2 = N2 / 16;
    static constexpr int FPC = N2 >= 1024 ? 4 : (SPX_K2_THREADS_B / T2 > 32 ? 32 : SPX_K2_THREADS_B / T2);  // rows per CTA
    static constexpr int THREADS_B = FPC * T2;
    static constexpr int P2 = plan_passes(N2);
    static constexpr int BUF2 = padded_size(N2) + (P2 >= 3 ? N2 : 0);
    static constexpr int TW2 = plan_tw_size(N2);
    static constexpr int TILE_LD = FPC + 1;                    // padded tile row (floats)
    // shared memory (bytes): [exchange buffers][twiddle table][staging of the next frame][dB tile (B only)]
    static constexpr size_t smem_a(int elt) { return (size_t)(G * S1 + TW1) * 8 + (size_t)N1 * G * elt; }
    static constexpr size_t smem_b() { return (size_t)(FPC * BUF2 + TW2) * 8 + (size_t)FPC * N2 * 8 + (size_t)N2 * TILE_LD * 4; }
};

// Prefetch of the next frame, two flavours (template parameter TMA):
//   TMA  : bulk asynchronous copies (cp.async.bulk + mbarrier, SASS UBLKCP) -- one 128-byte row segment per thread in
//          kernel A, one whole row per slot in kernel B; issued after the frame's first barrier (every thread has read
//          the staging buffer by then).  Needs 16-byte aligned segments.
//   !TMA : cp.async (LDGSTS) where every thread prefetches exactly the elements it will read back itself, so the
//          staging buffer needs no barrier; used when frame starts are not 16-byte aligned.
// ------------------------------------------------------------------ kernel A: column FFTs + twiddle
// A CTA owns one group of G adjacent columns for all its frames (grid = groups x frame lanes), so the window
// values and the W_N^{n2 k1} twiddles of a thread are frame-invariant and live in registers.
#ifndef SPX_K2_OCC_A
#define SPX_K2_OCC_A 1
#endif
template <int N1, int N2, int FMT, bool TMA>
__global__ void __launch_bounds__(BigCfg<N1, N2>::THREADS_A, (BigCfg<N1, N2>::THREADS_A <= 256 ? SPX_K2_OCC_A : 1))
big_cols_kernel(const BigParams p) {
    using C = BigCfg<N1, N2>;
    constexpr int N = C::N, T1 = C::T1, G = C::G, P = C::P1;
    constexpr int ELT = FMT == FMT_CF32 ? 8 : 4;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* smem = reinterpret_cast<float2*>(smem_raw);
    float2* tws = smem + G * C::S1;
    unsigned char* stage = smem_raw + (size_t)(G * C::S1 + C::TW1) * 8;
    const int c = threadIdx.x % G;     // column inside the group (fast lane index -> coalesced rows)
    const int tid = threadIdx.x / G;   // position inside the N1-point FFT
    float2* bufA = smem + c * C::S1;
    float2* bufB = bufA + padded_size(N1);
    constexpr int GROUPS = N2 / G;
    const int g = blockIdx.x % GROUPS;
    const int lane_f = blockIdx.x / GROUPS, lanes_f = gridDim.x / GROUPS;   // host: gridDim.x is a multiple of GROUPS
    const int n2 = g * G + c;
    for (int i = threadIdx.x; i < C::TW1; i += C::THREADS_A) tws[i] = __ldg(p.tw1 + i);

    constexpr int SL = P - 1, RL = plan_radix(N1, SL), NB = 16 / RL;
    float w[16];
    float2 wn[16];
#pragma unroll
    for (int t = 0; t < 16; ++t) w[t] = p.win ? __ldg(p.win + N2 * (tid + t * T1) + n2) : 1.0f;
#pragma unroll
    for (int u = 0; u < NB; ++u)
#pragma unroll
        for (int t = 0; t < RL; ++t) {
            const int k1 = tid + T1 * u + t * (N1 / RL);
            const unsigned m = ((unsigned)n2 * (unsigned)k1) & (unsigned)(N - 1);
            wn[u * RL + t] = cmul(__ldg(p.wn_coarse + (m >> 8)), __ldg(p.wn_fine + (m & 255u)));
        }
    const char* in_bytes = reinterpret_cast<const char*>(p.in);
    __shared__ unsigned long long mbar_a;
    const unsigned bar_u32 = smem_u32(&mbar_a);
    const unsigned stage_u32 = smem_u32(stage);
    auto prefetch = [&](int f) {
        if constexpr (TMA) {
            // one bulk copy per row segment (G columns = G*ELT bytes), rows spread over the CTA's threads
            const char* src0 = in_bytes + (size_t)(p.sample0 + (long long)f * p.hop + g * G) * ELT;
            if (threadIdx.x == 0) mbar_expect_tx(bar_u32, (unsigned)(N1 * G * ELT));
            for (int row = threadIdx.x; row < N1; row += C::THREADS_A)
                bulk_g2s(stage_u32 + (unsigned)(row * G * ELT), src0 + (size_t)N2 * row * ELT, (unsigned)(G * ELT), bar_u32);
        } else {
            const char* src = in_bytes + (size_t)(p.sample0 + (long long)f * p.hop + n2) * ELT;
#pragma unroll
            for (int t = 0; t < 16; ++t) {
                const int row = tid + t * T1;
                if (FMT == FMT_CF32) cp_async8(stage + (size_t)(row * G + c) * ELT, src + (size_t)N2 * row * ELT);
                else                 cp_async4(stage + (size_t)(row * G + c) * ELT, src + (size_t)N2 * row * ELT);
            }
        }
    };
    if constexpr (TMA) {
        if (threadIdx.x == 0) mbar_init(bar_u32, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        __syncthreads();
    }
    if (lane_f < p.frames) prefetch(lane_f);
    __syncthreads();  // twiddle table visible
    unsigned parity = 0;
    float2 v[16];
    for (int f = lane_f; f < p.frames; f += lanes_f) {
        if constexpr (TMA) { mbar_wait(bar_u32, parity); parity ^= 1u; }
        else cp_async_wait_all();
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            const int row = tid + t * T1;
            float2 x;
            if (FMT == FMT_CF32) x = reinterpret_cast<const float2*>(stage)[row * G + c];
            else                 x = ci16_to_f2<TUNE_I2FP>(reinterpret_cast<const unsigned int*>(stage)[row * G + c]);
            v[t] = make_float2(x.x * w[t], x.y * w[t]);
        }
        const bool more = f + lanes_f < p.frames;
        if constexpr (!TMA) { if (more) prefetch(f + lanes_f); }   // own slots only: overlaps the whole transform below
        pass_dft<N1, 0>(v);
        if constexpr (P > 1) {
            pass_store_smem<N1, 0>(v, tid, bufA);
            __syncthreads();
            if constexpr (TMA) { if (more) prefetch(f + lanes_f); }   // every thread has read the staging tile
            pass_load_smem<N1, 1>(v, tid, bufA);
            pass_twiddle_table<N1, 1, true>(v, tid, tws);
            pass_dft<N1, 1>(v);
        }
        if constexpr (P > 2) {
            pass_store_smem<N1, 1>(v, tid, bufB);
            __syncthreads();
            pass_load_smem<N1, 2>(v, tid, bufB);
            pass_twiddle_table<N1, 2, true>(v, tid, tws);
            pass_dft<N1, 2>(v);
        }
        static_assert(P <= 3, "N1 up to 4096");
        // twiddle W_N^{n2*k1} and store T[k1][n2]
        float2* trow = p.scratch + (long long)f * N + n2;
#pragma unroll
        for (int u = 0; u < NB; ++u)
#pragma unroll
            for (int t = 0; t < RL; ++t) {
                const int k1 = tid + T1 * u + t * (N1 / RL);
                trow[(long long)k1 * N2] = cmul(v[u * RL + t], wn[u * RL + t]);
            }
        if constexpr (P > 1) __syncthreads();  // exchange buffers are rewritten by the next frame
    }
}

// ------------------------------------------------------------------ kernel B: row FFTs + fused epilogue
template <int N1, int N2, bool ACC, bool TMA>
__global__ void __launch_bounds__(BigCfg<N1, N2>::THREADS_B) big_rows_kernel(const BigParams p) {
    using C = BigCfg<N1, N2>;
    constexpr int N = C::N, T2 = C::T2, FPC = C::FPC, P = C::P2, LD = C::TILE_LD;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* smem = reinterpret_cast<float2*>(smem_raw);
    float2* tws = smem + FPC * C::BUF2;
    float2* stage = tws + C::TW2;                                  // [FPC][N2] next frame's rows
    float* tile = reinterpret_cast<float*>(stage + FPC * N2);      // [N2][LD] log2-power tile for the transposed store
    const int slot = threadIdx.x / T2;
    const int tid = threadIdx.x - slot * T2;
    float2* bufA = smem + slot * C::BUF2;
    float2* bufB = bufA + padded_size(N2);
    float2* my_stage = stage + slot * N2;
    for (int i = threadIdx.x; i < C::TW2; i += C::THREADS_B) tws[i] = __ldg(p.tw2 + i);
    constexpr int GROUPS = N1 / FPC;
    const int chunks = (p.frames + p.frames_per_chunk - 1) / p.frames_per_chunk;
    const long long items = (long long)GROUPS * chunks;
    constexpr int SL = P - 1, RL = plan_radix(N2, SL), NB = 16 / RL;
    __shared__ unsigned long long mbar_b[FPC];
    const unsigned bar_u32 = smem_u32(&mbar_b[slot]);
    const unsigned my_stage_u32 = smem_u32(my_stage);
    auto prefetch = [&](long long it, int f) {   // rows of frame f for item `it` (its row group)
        const int gg = (int)(it % GROUPS);
        const float2* row = p.scratch + (long long)f * N + (long long)(gg * FPC + slot) * N2;
        if constexpr (TMA) {
            if (tid == 0) {   // one bulk copy per slot: its whole N2-point row
                mbar_expect_tx(bar_u32, (unsigned)(N2 * 8));
                bulk_g2s(my_stage_u32, row, (unsigned)(N2 * 8), bar_u32);
            }
        } else {
#pragma unroll
            for (int t = 0; t < 16; ++t) cp_async8(my_stage + tid + t * T2, row + tid + t * T2);
        }
    };
    if constexpr (TMA) {
        if (tid == 0) mbar_init(bar_u32, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        __syncthreads();
    }
    unsigned parity = 0;
    StftAcc<ACC> acc;
    acc.reset();
    float2 v[16];
    if ((long long)blockIdx.x < items) prefetch(blockIdx.x, (int)(blockIdx.x / GROUPS) * p.frames_per_chunk);
    __syncthreads();
    for (long long it = blockIdx.x; it < items; it += gridDim.x) {
        const int g = (int)(it % GROUPS);        // consecutive CTAs take consecutive row groups of the same frames
        const int ch = (int)(it / GROUPS);
        const int k1 = g * FPC + slot;
        const int f_lo = ch * p.frames_per_chunk;
        const int f_hi = min(p.frames, f_lo + p.frames_per_chunk);
        for (int f = f_lo; f < f_hi; ++f) {
            if constexpr (TMA) { mbar_wait(bar_u32, parity); parity ^= 1u; }
            else cp_async_wait_all();
#pragma unroll
            for (int t = 0; t < 16; ++t) v[t] = my_stage[tid + t * T2];
            // next frame of this item, or the first frame of this CTA's next item
            auto prefetch_next = [&]() {
                if (f + 1 < f_hi) prefetch(it, f + 1);
                else if (it + gridDim.x < items) prefetch(it + gridDim.x, (int)((it + gridDim.x) / GROUPS) * p.frames_per_chunk);
            };
            if constexpr (!TMA) prefetch_next();
            pass_dft<N2, 0>(v);
            if constexpr (P > 1) {
                pass_store_smem<N2, 0>(v, tid, bufA);
                __syncthreads();
                if constexpr (TMA) prefetch_next();   // every thread of the slot has read its staged row
                pass_load_smem<N2, 1>(v, tid, bufA);
                pass_twiddle_table<N2, 1, true>(v, tid, tws);
                pass_dft<N2, 1>(v);
            }
            if constexpr (P > 2) {
                pass_store_smem<N2, 1>(v, tid, bufB);
                __syncthreads();
                pass_load_smem<N2, 2>(v, tid, bufB);
                pass_twiddle_table<N2, 2, true>(v, tid, tws);
                pass_dft<N2, 2>(v);
            }
            static_assert(P <= 3, "N2 up to 4096");
            const long long orow = (p.row0 + f) * (long long)N;
            // bin k = k1 + N1*k2 -> fftshift position k1 + N1*((k2 + N2/2) mod N2)
            if (p.spec_rows) {
#pragma unroll
                for (int u = 0; u < NB; ++u)
#pragma unroll
                    for (int t = 0; t < RL; ++t) {
                        const int k2s = (tid + T2 * u + t * (N2 / RL) + N2 / 2) & (N2 - 1);
                        p.spec_rows[orow + k1 + (long long)N1 * k2s] = v[u * RL + t];
                    }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i].x = v[i].x * v[i].x + v[i].y * v[i].y;
            if (ACC) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    acc.sum[i] += v[i].x;
                    acc.mx[i] = fmaxf(acc.mx[i], v[i].x);
                }
            }
            if (p.db_rows || p.wf_rows) {
                // y = log2 of the (eps-corrected) power; one uniform branch per thread as in K1's epilogue
                float pmin = v[0].x;
#pragma unroll
                for (int i = 1; i < 16; ++i) pmin = fminf(pmin, v[i].x);
                if (pmin >= p.db_pw_min) {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i].y = fast_log2(v[i].x);
                } else {
#pragma unroll
                    for (int i = 0; i < 16; ++i) v[i].y = 2.0f * fast_log2(fast_sqrt(v[i].x) + p.db_eps);
                }
#pragma unroll
                for (int u = 0; u < NB; ++u)
#pragma unroll
                    for (int t = 0; t < RL; ++t) {
                        const int k2s = (tid + T2 * u + t * (N2 / RL) + N2 / 2) & (N2 - 1);
                        tile[k2s * LD + slot] = v[u * RL + t].y;
                    }
                __syncthreads();
                // copy out: for every k2 a run of FPC consecutive bins k1_0 .. k1_0+FPC-1, written as 8-bin vectors
                const int k1_0 = g * FPC;
                constexpr int VW = FPC >= 8 ? 8 : 4, NV = FPC / VW;
                for (int idx = threadIdx.x; idx < N2 * NV; idx += C::THREADS_B) {
                    const int j0 = (idx % NV) * VW, k2s = idx / NV;
                    float y[VW];
#pragma unroll
                    for (int q = 0; q < VW; ++q) y[q] = tile[k2s * LD + j0 + q];
                    const long long o = orow + k1_0 + j0 + (long long)N1 * k2s;
                    if (p.db_rows) {
                        constexpr float K = 0.5f * SPX_DB_PER_LOG2;
#pragma unroll
                        for (int q = 0; q < VW; q += 4)
                            *reinterpret_cast<float4*>(p.db_rows + o + q) = make_float4(K * y[q], K * y[q + 1], K * y[q + 2], K * y[q + 3]);
                    }
                    if (p.wf_rows) {
                        unsigned int wd[VW / 4];
#pragma unroll
                        for (int h = 0; h < VW / 4; ++h) {
                            wd[h] = 0u;
#pragma unroll
                            for (int q = 0; q < 4; ++q) wd[h] |= sat_floor_u8(quant_pre(y[4 * h + q], p.q_a, p.q_b)) << (8 * q);
                        }
                        if constexpr (VW == 8) *reinterpret_cast<uint2*>(p.wf_rows + o) = make_uint2(wd[0], wd[1]);
                        else *reinterpret_cast<unsigned int*>(p.wf_rows + o) = wd[0];
                    }
                }
                // no barrier here: the next write of `tile` comes after the next frame's exchange barrier
            }
            if constexpr (P > 1) __syncthreads();  // exchange buffers (and the tile) are reused by the next frame
        }
        if constexpr (ACC) {
#pragma unroll
            for (int u = 0; u < NB; ++u)
#pragma unroll
                for (int t = 0; t < RL; ++t) {
                    const int k2s = (tid + T2 * u + t * (N2 / RL) + N2 / 2) & (N2 - 1);
                    const long long o = k1 + (long long)N1 * k2s;
                    flush_acc(p.welch_acc, p.maxhold, o, acc.sum[u * RL + t], acc.mx[u * RL + t], p.sys_atomics);
                }
            acc.reset();
        }
    }
}

// ------------------------------------------------------------------ host side
static void split_n(int n, int* n1, int* n2) {
    int lg = 0;
    while ((1 << lg) < n) ++lg;
    *n1 = 1 << (lg / 2);
    *n2 = n / *n1;
}

int bigfft_plan_init(spx_plan* pl) {
    const int n = pl->cfg.nfft;
    int n1, n2;
    split_n(n, &n1, &n2);
    pl->big_n1 = n1;
    pl->big_n2 = n2;
    std::vector<float2> t1 = build_twiddles(n1), t2 = build_twiddles(n2);
    std::vector<float2> fine(256), coarse((size_t)n / 256);
    const double two_pi = 6.283185307179586476925286766559;
    for (int i = 0; i < 256; ++i) {
        const double a = -two_pi * (double)i / (double)n;
        fine[i] = make_float2((float)cos(a), (float)sin(a));
    }
    for (int i = 0; i < n / 256; ++i) {
        const double a = -two_pi * (double)i * 256.0 / (double)n;
        coarse[i] = make_float2((float)cos(a), (float)sin(a));
    }
    const size_t total = t1.size() + t2.size() + fine.size() + coarse.size();
    SPX_CUDA(cudaMalloc(&pl->d_big_tw, total * sizeof(float2)));
    float2* d = pl->d_big_tw;
    pl->d_tw1 = d;
    SPX_CUDA(cudaMemcpy(d, t1.data(), t1.size() * sizeof(float2), cudaMemcpyHostToDevice));
    d += t1.size();
    pl->d_tw2 = d;
    SPX_CUDA(cudaMemcpy(d, t2.data(), t2.size() * sizeof(float2), cudaMemcpyHostToDevice));
    d += t2.size();
    pl->d_wn_fine = d;
    SPX_CUDA(cudaMemcpy(d, fine.data(), fine.size() * sizeof(float2), cudaMemcpyHostToDevice));
    d += fine.size();
    pl->d_wn_coarse = d;
    SPX_CUDA(cudaMemcpy(d, coarse.data(), coarse.size() * sizeof(float2), cudaMemcpyHostToDevice));
    return SPX_OK;
}

// what runs between the two kernels of a pair: order the row kernel (stream st) behind the column kernel (stream sa)
struct BigOrder {
    cudaStream_t sa;
    cudaEvent_t a_done;   // recorded on sa after the column kernel; st waits for it (nullptr: same stream, no event)
};

template <int N1, int N2, bool TMA_A>
static int big_launch_pair_t(spx_plan* pl, BigParams& p, cudaStream_t st, bool acc, bool cf32, const BigOrder& ord);

template <int N1, int N2>
static int big_launch_pair(spx_plan* pl, BigParams& p, cudaStream_t st, const BigOrder& ord) {
    const bool acc = p.welch_acc != nullptr || p.maxhold != nullptr;
    const bool cf32 = pl->cfg.in_fmt == SPX_FMT_CF32;
    // bulk copies need 16-byte aligned row segments: every frame start must be 16-byte aligned
    const size_t elt = cf32 ? 8 : 4;
    const bool tma_a = ((uintptr_t)p.in & 15u) == 0 && ((size_t)p.hop * elt) % 16 == 0 && ((size_t)p.sample0 * elt) % 16 == 0;
    return tma_a ? big_launch_pair_t<N1, N2, true>(pl, p, st, acc, cf32, ord) : big_launch_pair_t<N1, N2, false>(pl, p, st, acc, cf32, ord);
}

template <int N1, int N2, bool TMA_A>
static int big_launch_pair_t(spx_plan* pl, BigParams& p, cudaStream_t st, bool acc, bool cf32, const BigOrder& ord) {
    using C = BigCfg<N1, N2>;
    const size_t smem_a = C::smem_a(cf32 ? 8 : 4);
    const size_t smem_b = C::smem_b();
    auto ka_c = big_cols_kernel<N1, N2, FMT_CF32, TMA_A>;
    auto ka_i = big_cols_kernel<N1, N2, FMT_CI16, TMA_A>;
    auto kb_a = big_rows_kernel<N1, N2, true, true>;    // the scratch rows are always 16-byte aligned
    auto kb_n = big_rows_kernel<N1, N2, false, true>;
    int occ_cols[2] = {0, 0}, occ_rows[2] = {0, 0};   // kernel A: cf32, ci16 input; kernel B: with, without accumulators
    SPX_TRY(kernel_setup((const void*)ka_c, C::THREADS_A, C::smem_a(8), &occ_cols[0]));
    SPX_TRY(kernel_setup((const void*)ka_i, C::THREADS_A, C::smem_a(4), &occ_cols[1]));
    SPX_TRY(kernel_setup((const void*)kb_a, C::THREADS_B, smem_b, &occ_rows[0]));
    SPX_TRY(kernel_setup((const void*)kb_n, C::THREADS_B, smem_b, &occ_rows[1]));
    if (occ_cols[0] < 1 || occ_cols[1] < 1 || occ_rows[0] < 1 || occ_rows[1] < 1)
        return spx_set_error(SPX_E_CUDA, "large-N kernel does not fit on an SM (N1=%d N2=%d)", N1, N2);
    // kernel A: grid = column groups x frame lanes (a multiple of the group count: a CTA keeps its columns)
    constexpr int GROUPS_A = N2 / C::G;
    const int resident_a = pl->sm_count * occ_cols[cf32 ? 0 : 1];
    int lanes = resident_a / GROUPS_A;
    if (lanes < 1) lanes = 1;
    if (lanes > p.frames) lanes = p.frames;
    const unsigned grid_a = (unsigned)(GROUPS_A * lanes);
    if (cf32) ka_c<<<grid_a, C::THREADS_A, smem_a, ord.sa>>>(p);
    else ka_i<<<grid_a, C::THREADS_A, smem_a, ord.sa>>>(p);
    SPX_CUDA(cudaGetLastError());
    if (ord.a_done) {
        SPX_CUDA(cudaEventRecord(ord.a_done, ord.sa));
        SPX_CUDA(cudaStreamWaitEvent(st, ord.a_done, 0));
    }
    // kernel B: (row groups) x (frame chunks) work items, one resident wave; accumulators flush once per item
    const int groups = N1 / C::FPC;
    const int resident_b = pl->sm_count * occ_rows[acc ? 0 : 1];
    int chunks = (resident_b + groups - 1) / groups;
    if (chunks > p.frames) chunks = p.frames;
    if (chunks < 1) chunks = 1;
    p.frames_per_chunk = (p.frames + chunks - 1) / chunks;
    const long long items_b = (long long)groups * ((p.frames + p.frames_per_chunk - 1) / p.frames_per_chunk);
    const long long grid_b = items_b < resident_b ? items_b : resident_b;
    if (acc) kb_a<<<(unsigned)grid_b, C::THREADS_B, smem_b, st>>>(p);
    else kb_n<<<(unsigned)grid_b, C::THREADS_B, smem_b, st>>>(p);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

// one stream, frames [0, frames): batches of frames through the L2-sized scratch
int bigfft_launch_stream(spx_plan* pl, const void* in, long long frames, long long row0, const StftOut& out, cudaStream_t st) {
    const int n = pl->cfg.nfft;
    if (big2_eligible(pl, in, out))   // config-5 shape: one persistent kernel, scratch stays in L2
        return big2_launch_stream(pl, in, frames, row0, out, st);
    const size_t frame_bytes = (size_t)n * sizeof(float2);
    // two halves of the scratch: the column kernel of batch k+1 (aux stream) runs next to the row kernel of batch k, so
    // the tail wave of one kernel is filled by the other instead of leaving SMs idle
    long long fb = (long long)(pl->big_scratch_bytes / 2 / frame_bytes);
    if (fb < 1) fb = 1;
    if (fb > frames) fb = frames;
    const bool two = frames > fb;
    SPX_TRY(pl->st_big.reserve((size_t)fb * frame_bytes * (two ? 2 : 1)));
    if (two && !pl->s_big_aux) {
        SPX_CUDA(cudaStreamCreateWithFlags(&pl->s_big_aux, cudaStreamNonBlocking));
        for (cudaEvent_t& e : pl->ev_big) SPX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    BigParams p;
    memset(&p, 0, sizeof(p));
    p.in = in;
    p.hop = pl->cfg.hop;
    p.win = pl->d_win;
    p.tw1 = pl->d_tw1;
    p.tw2 = pl->d_tw2;
    p.wn_fine = pl->d_wn_fine;
    p.wn_coarse = pl->d_wn_coarse;
    p.db_rows = out.db;
    p.wf_rows = out.wf;
    p.spec_rows = out.spec;
    p.welch_acc = out.welch;
    p.maxhold = out.maxhold;
    p.db_eps = pl->cfg.db_eps;
    p.db_pw_min = db_pw_min(pl);
    p.q_a = out.q_a();
    p.q_b = out.q_b();
    p.sys_atomics = out.sys_atomics;
    if (two) {   // everything already queued on st (accumulator memsets, the previous call) comes first
        SPX_CUDA(cudaEventRecord(pl->ev_big[0], st));
        SPX_CUDA(cudaStreamWaitEvent(pl->s_big_aux, pl->ev_big[0], 0));
    }
    long long k = 0;
    for (long long f0 = 0; f0 < frames; f0 += fb, ++k) {
        const int b = (int)(k & 1);
        p.frames = (int)(frames - f0 < fb ? frames - f0 : fb);
        p.sample0 = f0 * pl->cfg.hop;
        p.row0 = row0 + f0;
        p.scratch = (float2*)pl->st_big.ptr + (size_t)(two ? b : 0) * (size_t)fb * n;
        BigOrder ord{st, nullptr};
        if (two) {
            ord.sa = pl->s_big_aux;
            ord.a_done = pl->ev_big[1 + b];
            if (k >= 2) SPX_CUDA(cudaStreamWaitEvent(pl->s_big_aux, pl->ev_big[3 + b], 0));   // rows of batch k-2 left this half
        }
        int rc;
        switch (n) {
            case 1 << 14: rc = big_launch_pair<128, 128>(pl, p, st, ord); break;
            case 1 << 15: rc = big_launch_pair<128, 256>(pl, p, st, ord); break;
            case 1 << 16: rc = big_launch_pair<256, 256>(pl, p, st, ord); break;
            case 1 << 17: rc = big_launch_pair<256, 512>(pl, p, st, ord); break;
            case 1 << 18: rc = big_launch_pair<512, 512>(pl, p, st, ord); break;
            case 1 << 19: rc = big_launch_pair<512, 1024>(pl, p, st, ord); break;
            case 1 << 20: rc = big_launch_pair<1024, 1024>(pl, p, st, ord); break;
            default: return spx_set_error(SPX_E_UNSUPPORTED, "nfft %d", n);
        }
        SPX_TRY(rc);
        if (two) SPX_CUDA(cudaEventRecord(pl->ev_big[3 + b], st));
    }
    return SPX_OK;
}

}  // namespace spx
