// spx_stft_kernel.cuh -- K1: the fused STFT kernel and its launcher template.
//
// Persistent CTAs; each CTA hosts FPC "slots" of T = N/16 threads, one frame in flight per slot.
// A slot walks chunks of consecutive frames of one stream, keeps the Welch sum and max-hold of
// its 16 bins per thread in registers, and flushes them with fp64 / ordered-uint atomics at the
// end of every chunk.  Rows (f32 dB, u8, complex) are written straight from the registers of the
// last FFT pass in fftshift order.
#pragma once
#include "spx_stft_device.cuh"
#include "spx_async.cuh"
#include "spx_internal.h"

namespace spx {

template <int N>
struct StftCfg {
    static constexpr int T = N / 16;
    static constexpr int FPC = (T >= 256) ? 1 : 256 / T;
    static constexpr int THREADS = T * FPC;
    static constexpr int P = plan_passes(N);
    static constexpr int BUF_F2 = (P >= 2 ? padded_size(N) : 0) + (P >= 3 ? N : 0);  // exchange buffers per slot
    static constexpr int TW_F2 = plan_tw_size(N);
    static constexpr bool CAN_STAGE = T >= 32;  // one elected lane per slot issues the bulk copy
    // float2 per slot including the staging area for one raw frame (cf32: N float2, ci16: N/2 float2)
    __host__ __device__ static constexpr int slot_f2(bool stage, int fmt) { return BUF_F2 + (stage ? (fmt == FMT_CF32 ? N : N / 2) : 0); }
    // staged kernels also keep half of the symmetric window in shared memory (N/2 floats = N/4 float2), once per CTA
    __host__ __device__ static constexpr int win_f2(bool stage) { return stage ? N / 4 : 0; }
};

// barrier among the T threads of one slot; slots never wait for each other
template <int N>
__device__ __forceinline__ void slot_barrier(int slot) {
    using C = StftCfg<N>;
    if constexpr (C::FPC == 1) {
        __syncthreads();
    } else if constexpr (C::T >= 32) {
        asm volatile("bar.sync %0, %1;" ::"r"(slot + 1), "n"(C::T) : "memory");
    } else {
        // several slots share a warp: synchronise exactly this slot's lanes
        const unsigned lane0 = (threadIdx.x & 31u) & ~(unsigned)(C::T - 1);
        const unsigned mask = (C::T >= 32 ? 0xffffffffu : ((1u << C::T) - 1u)) << lane0;
        __syncwarp(mask);
    }
}

// position of a worker (slot) in its frame sequence: chunks worker, worker + n_workers, ...
struct FrameCursor {
    unsigned chunk;
    int fi, nf;
    unsigned stream;
    long long sbase, rbase;  // first sample / first row of the chunk
    bool valid;
    __device__ __forceinline__ void seek(const StftParams& p, unsigned c) {
        chunk = c;
        valid = (long long)c < p.total_chunks;
        fi = 0;
        if (!valid) { nf = 0; stream = 0; sbase = 0; rbase = 0; return; }
        stream = c / (unsigned)p.chunks_per_stream;
        const long long f0 = (long long)(c - stream * (unsigned)p.chunks_per_stream) * p.frames_per_chunk;
        const long long left = p.frames_per_stream - f0;
        nf = (int)(left < p.frames_per_chunk ? left : p.frames_per_chunk);
        sbase = (long long)stream * p.stream_stride + f0 * p.hop;
        rbase = (long long)stream * p.frames_per_stream + f0;
    }
    __device__ __forceinline__ long long sample0(const StftParams& p) const { return sbase + (long long)fi * p.hop; }
    __device__ __forceinline__ long long row() const { return rbase + fi; }
};

template <int N, int FMT, bool ACC, int TWM, int OCC, bool STAGE, int TUNE = 0>
__global__ void __launch_bounds__(StftCfg<N>::THREADS, OCC) stft_kernel(const StftParams p) {
    using C = StftCfg<N>;
    constexpr int P = C::P;
    constexpr unsigned FRAME_BYTES = (unsigned)N * (FMT == FMT_CF32 ? 8u : 4u);
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ unsigned long long mbar[STAGE ? C::FPC : 1];
    float2* smem = reinterpret_cast<float2*>(smem_raw);

    const int slot = threadIdx.x / C::T;
    const int tid = threadIdx.x - slot * C::T;
    float2* slot_base = smem + slot * C::slot_f2(STAGE, FMT);
    void* stage = STAGE ? (void*)slot_base : nullptr;
    float2* bufA = slot_base + (STAGE ? (FMT == FMT_CF32 ? N : N / 2) : 0);
    float2* bufB = bufA + padded_size(N);

    const float2* tw = p.tw;
    const float* win_half = nullptr;
    if constexpr (STAGE) {
        if (p.win != nullptr) {
            float* wsm = reinterpret_cast<float*>(smem + C::FPC * C::slot_f2(STAGE, FMT));
            for (int i = threadIdx.x; i < N / 2; i += C::THREADS) wsm[i] = __ldg(p.win + i);
            win_half = wsm;
        }
    }
    constexpr bool TW_IN_SMEM = TWM == TW_SMEM && P > 1;
    if constexpr (TW_IN_SMEM) {
        float2* tws = smem + C::FPC * C::slot_f2(STAGE, FMT) + C::win_f2(STAGE);
        for (int i = threadIdx.x; i < C::TW_F2; i += C::THREADS) tws[i] = __ldg(p.tw + i);
        tw = tws;
    }
    const unsigned bar_u32 = smem_u32(&mbar[STAGE ? slot : 0]);
    const unsigned stage_u32 = smem_u32(slot_base);
    if constexpr (STAGE) {
        if (tid == 0) mbar_init(bar_u32, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if constexpr (STAGE || TW_IN_SMEM) __syncthreads();

    TwRegs<N> twr;
    if constexpr (TWM == TW_REG && P > 1) {
        tw_regs_load_pass<N, 1>(twr, tid, p.tw);
        if constexpr (P > 2) tw_regs_load_pass<N, 2>(twr, tid, p.tw);
        if constexpr (P > 3) tw_regs_load_pass<N, 3>(twr, tid, p.tw);
    }

    StftAcc<ACC> acc;
    acc.reset();

    const unsigned worker = blockIdx.x * C::FPC + slot;
    const unsigned n_workers = gridDim.x * C::FPC;
    const char* in_bytes = reinterpret_cast<const char*>(p.in);

    FrameCursor cur;
    cur.seek(p, worker);
    unsigned parity = 0;
    if constexpr (STAGE) {
        if (cur.valid && tid == 0) {
            mbar_expect_tx(bar_u32, FRAME_BYTES);
            bulk_g2s(stage_u32, in_bytes + cur.sample0(p) * (FMT == FMT_CF32 ? 8 : 4), FRAME_BYTES, bar_u32);
        }
    }

    float2 v[16];
    while (cur.valid) {
        const long long s0 = cur.sample0(p), row = cur.row();
        const bool last_in_chunk = cur.fi + 1 == cur.nf;
        const unsigned this_stream = cur.stream;
        // where the next frame of this slot lives (same chunk, or the slot's next chunk)
        FrameCursor nxt = cur;
        if (!last_in_chunk) nxt.fi = cur.fi + 1;
        else nxt.seek(p, cur.chunk + n_workers);

        if constexpr (STAGE) {
            mbar_wait(bar_u32, parity);
            parity ^= 1u;
        }
        stft_phase<N, FMT, ACC, TWM, 0, TUNE>(v, tid, p, s0, row, true, bufA, bufB, tw, twr, acc, stage, win_half);
        if constexpr (P > 1 || STAGE) slot_barrier<N>(slot);
        if constexpr (STAGE) {
            // every thread of the slot has read its staged samples: refill the buffer with the next frame
            if (nxt.valid && tid == 0) {
                mbar_expect_tx(bar_u32, FRAME_BYTES);
                bulk_g2s(stage_u32, in_bytes + nxt.sample0(p) * (FMT == FMT_CF32 ? 8 : 4), FRAME_BYTES, bar_u32);
            }
        }
        if constexpr (P > 1) stft_phase<N, FMT, ACC, TWM, 1>(v, tid, p, s0, row, true, bufA, bufB, tw, twr, acc);
        if constexpr (P > 2) {
            slot_barrier<N>(slot);
            stft_phase<N, FMT, ACC, TWM, 2>(v, tid, p, s0, row, true, bufA, bufB, tw, twr, acc);
        }
        if constexpr (P > 3) {
            slot_barrier<N>(slot);
            stft_phase<N, FMT, ACC, TWM, 3>(v, tid, p, s0, row, true, bufA, bufB, tw, twr, acc);
        }
        // the last pass of an even-P plan reads bufA, which the next frame's pass 0 overwrites
        if constexpr (P > 1 && (P % 2) == 0) slot_barrier<N>(slot);

        if constexpr (ACC) {
            if (last_in_chunk) {
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const long long o = (long long)this_stream * N + acc_pos<N>(tid, i);
                    flush_acc(p.welch_acc, p.maxhold, o, acc.sum[i], acc.mx[i], p.sys_atomics);
                }
                acc.reset();
            }
        }
        cur = nxt;
    }
}

// ------------------------------------------------------------------ host side
struct StftLaunch {
    StftParams p;          // chunking fields are filled in by the launcher
    int nfft;
    int in_fmt;
    int variant;           // spx_plan_config.variant: 0, or 12 / 22 to force K1 / the generic K1v2 kernel
    int sm_count;
    long long total_frames;  // n_streams * F
    cudaStream_t stream;
};

template <int N, int FMT, bool ACC, int TWM, int OCC, bool STAGE, int TUNE = 0>
int launch_stft_inst(StftLaunch& L) {
    using C = StftCfg<N>;
    auto kern = stft_kernel<N, FMT, ACC, TWM, OCC, STAGE, TUNE>;
    size_t smem = (size_t)(C::FPC * C::slot_f2(STAGE, FMT) + C::win_f2(STAGE)) * sizeof(float2);
    if (TWM == TW_SMEM) smem += (size_t)C::TW_F2 * sizeof(float2);
    int occ = 0;
    SPX_TRY(kernel_setup((const void*)kern, C::THREADS, smem, &occ));
    if (occ < 1) return spx_set_error(SPX_E_CUDA, "stft kernel does not fit on an SM");
    const long long workers_max = (long long)L.sm_count * occ * C::FPC;
    // chunking: <= 256 frames per chunk, chunks never cross a stream
    const long long F = L.p.frames_per_stream;
    long long per_worker = (L.total_frames + workers_max - 1) / workers_max;
    long long fpc = per_worker < 1 ? 1 : per_worker;
    if (fpc > 256) {
        const long long waves = (per_worker + 255) / 256;
        fpc = (per_worker + waves - 1) / waves;
    }
    if (fpc > F) fpc = F;
    const long long cps = (F + fpc - 1) / fpc;
    L.p.frames_per_chunk = (int)fpc;
    L.p.chunks_per_stream = (int)cps;
    L.p.total_chunks = cps * L.p.n_streams;
    long long grid = (L.p.total_chunks + C::FPC - 1) / C::FPC;
    const long long grid_max = (long long)L.sm_count * occ;
    if (grid > grid_max) grid = grid_max;
    if (grid < 1) grid = 1;
    kern<<<(unsigned)grid, C::THREADS, smem, L.stream>>>(L.p);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

// bulk async copies need 16-byte aligned source addresses and sizes: every frame start must be aligned
inline bool stage_ok(const StftLaunch& L) {
    const long long elt = L.in_fmt == FMT_CF32 ? 8 : 4;
    if (((uintptr_t)L.p.in & 15u) != 0) return false;
    if ((L.p.hop * elt) % 16 != 0) return false;
    if (L.p.n_streams > 1 && (L.p.stream_stride * elt) % 16 != 0) return false;
    return true;
}

// ACCS: which accumulator instances to build.  ACC_ANY picks at run time; a caller that has already branched on the
// accumulators passes ACC_OFF / ACC_ON so that the other instance, which it can never launch, is not compiled.
enum { ACC_ANY = 0, ACC_OFF = 1, ACC_ON = 2 };

template <int N, int FMT, int TWM, int OCC, bool STAGE, int TUNE, int ACCS>
int launch_stft_acc(StftLaunch& L) {
    if constexpr (ACCS == ACC_ANY) {
        const bool acc = L.p.welch_acc != nullptr || L.p.maxhold != nullptr;
        return acc ? launch_stft_inst<N, FMT, true, TWM, OCC, STAGE, TUNE>(L)
                   : launch_stft_inst<N, FMT, false, TWM, OCC, STAGE, TUNE>(L);
    } else {
        return launch_stft_inst<N, FMT, ACCS == ACC_ON, TWM, OCC, STAGE, TUNE>(L);
    }
}

template <int N, int TWM, int OCC, bool STAGE, int TUNE = 0, int ACCS = ACC_ANY>
int launch_stft_fmt(StftLaunch& L) {
    if (L.in_fmt == FMT_CF32) return launch_stft_acc<N, FMT_CF32, TWM, OCC, STAGE, TUNE, ACCS>(L);
    return launch_stft_acc<N, FMT_CI16, TWM, OCC, STAGE, TUNE, ACCS>(L);
}

// STAGE_WANTED: use the TMA-staged kernel when the input is suitably aligned, else direct loads
template <int N, int TWM, int OCC, bool STAGE_WANTED = false, int TUNE = 0, int ACCS = ACC_ANY>
int launch_stft_n(StftLaunch& L) {
    if constexpr (STAGE_WANTED && StftCfg<N>::CAN_STAGE) {
        if (stage_ok(L)) return launch_stft_fmt<N, TWM, OCC, true, TUNE, ACCS>(L);
    }
    return launch_stft_fmt<N, TWM, OCC, false, TUNE, ACCS>(L);
}

// one translation unit per size group instantiates these
int launch_stft_small(StftLaunch& L);   // N = 16 .. 512
int launch_stft_1k2k(StftLaunch& L);    // N = 1024, 2048
int launch_stft_4k(StftLaunch& L);      // N = 4096
int launch_stft_8k(StftLaunch& L);      // N = 8192

}  // namespace spx
