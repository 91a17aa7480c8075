// spx_stft2_kernel.cuh -- K1v2: fused STFT kernel with a warp-local first exchange and ONE block barrier per frame
// (phases in spx_stft2_device.cuh), N = 1024 / 2048 / 4096.
//
// Input staging is a 2-D TMA tensor copy (cp.async.bulk.tensor, SASS UTMALDG) of the frame viewed as rows of 128 bytes
// with CU_TENSOR_MAP_SWIZZLE_128B: phase A reads the frame with a stride of 16 C samples between registers and C
// samples between lanes, which would be a 16-way bank conflict on a linear copy; the hardware swizzle spreads the
// eight rows a half-warp touches over all banks.  The tensor map describes the caller's whole input buffer; it is
// encoded on the host per launch (a few hundred nanoseconds) and passed as a __grid_constant__ kernel parameter.
#pragma once
#include <cuda.h>
#include <stdlib.h>

#include "spx_stft2_device.cuh"
#include "spx_stft_kernel.cuh"

namespace spx {

template <int N, int FMT>
struct Stft2Cfg {
    using G = Stft2Geom<N>;
    static constexpr int T = G::T;
    static constexpr int FPC = 256 / T;                      // frames in flight per CTA (slots)
    static constexpr int THREADS = 256;
    static constexpr unsigned FRAME_BYTES = (unsigned)N * (FMT == FMT_CF32 ? 8u : 4u);
    static constexpr unsigned ROWS = FRAME_BYTES / 128u;     // box height of the tensor copy (<= 256)
    static constexpr size_t X_BYTES = (size_t)G::X_F2 * sizeof(float2);
    // [stage x FPC (1024-byte aligned)] [X0, X1 x FPC] [window table N/2 floats]  + 1024 bytes of alignment slack
    static constexpr size_t SMEM = (size_t)FPC * FRAME_BYTES + (size_t)FPC * 2 * X_BYTES + (size_t)(N / 2) * sizeof(float) + 1024;
};

__device__ __forceinline__ void tma_load_rows(unsigned dst, const CUtensorMap* tmap, int row, unsigned bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(tmap), "r"(0), "r"(row), "r"(bar)
                 : "memory");
}

template <int N, int FMT, bool ACC, int OCC, int TUNE>
__global__ void __launch_bounds__(256, OCC) stft2_kernel(const StftParams p, const __grid_constant__ CUtensorMap tmap) {
    using C = Stft2Cfg<N, FMT>;
    using G = Stft2Geom<N>;
    constexpr bool TWC_REGS = G::C == 16;
    constexpr int ELT = FMT == FMT_CF32 ? 8 : 4;
    extern __shared__ unsigned char smem_raw2[];
    __shared__ unsigned long long mbar[C::FPC];

    const int slot = threadIdx.x / C::T;
    const int tid = threadIdx.x - slot * C::T;
    // swizzled TMA destinations must sit on 1024-byte boundaries of the shared window
    const unsigned raw_u32 = smem_u32(smem_raw2);
    unsigned char* base = smem_raw2 + (((raw_u32 + 1023u) & ~1023u) - raw_u32);
    unsigned char* stage = base + (size_t)slot * C::FRAME_BYTES;
    float2* X0 = reinterpret_cast<float2*>(base + (size_t)C::FPC * C::FRAME_BYTES + (size_t)slot * 2 * C::X_BYTES);
    float2* X1 = X0 + G::X_F2;
    float* wtab = nullptr;
    if (p.win != nullptr) {
        wtab = reinterpret_cast<float*>(base + (size_t)C::FPC * C::FRAME_BYTES + (size_t)C::FPC * 2 * C::X_BYTES);
        if (slot == 0) k2_build_window<N>(wtab, p.win, tid);
    }
    const unsigned bar_u32 = smem_u32(&mbar[slot]);
    const unsigned stage_u32 = smem_u32(stage);
    if (tid == 0) mbar_init(bar_u32, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    TwRegs<N> twr;
    tw_regs_load_pass<N, 1>(twr, k2_ka_of(tid), p.tw);
    if constexpr (TWC_REGS) tw_regs_load_pass<N, 2>(twr, tid, p.tw);

    StftAcc<ACC> acc;
    acc.reset();

    const unsigned worker = blockIdx.x * C::FPC + slot;
    const unsigned n_workers = gridDim.x * C::FPC;
    FrameCursor cur;
    cur.seek(p, worker);
    unsigned parity = 0;
    if (cur.valid && tid == 0) {
        mbar_expect_tx(bar_u32, C::FRAME_BYTES);
        tma_load_rows(stage_u32, &tmap, (int)((cur.sample0(p) * ELT) >> 7), bar_u32);
    }

    float2 v[16];
    while (cur.valid) {
        const long long row = cur.row();
        const bool last_in_chunk = cur.fi + 1 == cur.nf;
        const unsigned this_stream = cur.stream;
        FrameCursor nxt = cur;
        if (!last_in_chunk) nxt.fi = cur.fi + 1;
        else nxt.seek(p, cur.chunk + n_workers);
        float2* X = parity ? X1 : X0;

        // TUNE_L2PF (the launcher picks it for cf32, N = 4096, hop >= N).  Non-overlapping frames come straight from HBM, and the
        // tensor copy of the next frame is only issued after this frame's barrier -- less than half a frame time to hide an HBM
        // access.  Ask L2 for the next frame now: its copy then has an L2 hit's latency (headline shape 0.745 -> 0.78 of HBM).
        // A compile-time switch: as a run-time branch it cost the overlapped int16 kernel 5 registers and 1.4 %.
        if constexpr ((TUNE & TUNE_L2PF) != 0) {
            if (tid == 0 && cur.fi + 1 < cur.nf) {
                const char* src = reinterpret_cast<const char*>(p.in) + (cur.sample0(p) + (long long)p.hop) * ELT;
                asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(C::FRAME_BYTES) : "memory");
            }
        }
        mbar_wait(bar_u32, parity);
        k2_phase_a<N, FMT, TUNE>(v, tid, stage, wtab, X);
        __syncwarp();
        k2_phase_b1<N, TUNE>(v, tid, X, twr);
        __syncwarp();
        k2_phase_b2<N>(v, tid, X);
        slot_barrier<N>(slot);          // the only block-level barrier of the frame
        // every thread of the slot has consumed the staged samples: refill the buffer with the next frame
        if (nxt.valid && tid == 0) {
            mbar_expect_tx(bar_u32, C::FRAME_BYTES);
            tma_load_rows(stage_u32, &tmap, (int)((nxt.sample0(p) * ELT) >> 7), bar_u32);
        }
        k2_phase_c<N, ACC, TWC_REGS, TUNE>(v, tid, X, p, row, p.tw, twr, acc);
        parity ^= 1u;

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

// ------------------------------------------------------------------ strip staging of overlapping frames
// N = 4096, hop = N / R: only the newest hop block of a frame crosses L2 -> shared memory (north_star: "TMA /
// shared-memory staging of overlapping frames").  Same arithmetic and data flow as stft2_kernel otherwise.
template <int FMT, bool ACC, int R, int OCC, int TUNE>
__global__ void __launch_bounds__(256, OCC) stft2_strip_kernel(const StftParams p, const __grid_constant__ CUtensorMap tmap) {
    constexpr int N = 4096;
    using C = Stft2Cfg<N, FMT>;
    using G = Stft2Geom<N>;
    constexpr int ELT = FMT == FMT_CF32 ? 8 : 4;
    constexpr unsigned BLK = C::FRAME_BYTES / R;
    extern __shared__ unsigned char smem_raw2[];
    __shared__ unsigned long long mbar;
    const int tid = threadIdx.x;
    const unsigned raw_u32 = smem_u32(smem_raw2);
    unsigned char* base = smem_raw2 + (((raw_u32 + 1023u) & ~1023u) - raw_u32);
    unsigned char* stage = base;
    float2* X0 = reinterpret_cast<float2*>(base + C::FRAME_BYTES);
    float2* X1 = X0 + G::X_F2;
    float* wtab = nullptr;
    if (p.win != nullptr) {
        wtab = reinterpret_cast<float*>(base + C::FRAME_BYTES + 2 * C::X_BYTES);
        k2_build_window<N>(wtab, p.win, tid);
    }
    const unsigned bar_u32 = smem_u32(&mbar), stage_u32 = smem_u32(stage);
    if (tid == 0) mbar_init(bar_u32, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    TwRegs<N> twr;
    tw_regs_load_pass<N, 1>(twr, k2_ka_of(tid), p.tw);
    tw_regs_load_pass<N, 2>(twr, tid, p.tw);
    StftAcc<ACC> acc;
    acc.reset();

    // elected thread: copy what frame `c` still lacks -- the whole frame (R blocks) at the start of a chunk, else its newest block
    auto fetch = [&](const FrameCursor& c) {
        const long long row0 = (c.sample0(p) * ELT) >> 7;
        if (c.fi == 0) {
            mbar_expect_tx(bar_u32, C::FRAME_BYTES);
#pragma unroll
            for (int j = 0; j < R; ++j) tma_load_rows(stage_u32 + j * BLK, &tmap, (int)(row0 + j * (BLK / 128)), bar_u32);
        } else {
            mbar_expect_tx(bar_u32, BLK);
            tma_load_rows(stage_u32 + (unsigned)((c.fi - 1) & (R - 1)) * BLK, &tmap, (int)(row0 + (R - 1) * (BLK / 128)), bar_u32);
        }
    };

    const unsigned n_workers = gridDim.x;
    FrameCursor cur;
    cur.seek(p, blockIdx.x);
    unsigned parity = 0;
    if (cur.valid && tid == 0) fetch(cur);
    float2 v[16];
    while (cur.valid) {
        const long long row = cur.row();
        const bool last_in_chunk = cur.fi + 1 == cur.nf;
        const unsigned this_stream = cur.stream;
        FrameCursor nxt = cur;
        if (!last_in_chunk) nxt.fi = cur.fi + 1;
        else nxt.seek(p, cur.chunk + n_workers);
        float2* X = parity ? X1 : X0;
        mbar_wait(bar_u32, parity);
        k2_phase_a_strip<FMT, R, TUNE>(v, tid, stage, cur.fi & (R - 1), wtab, X);
        __syncwarp();
        k2_phase_b1<N, TUNE>(v, tid, X, twr);
        __syncwarp();
        k2_phase_b2<N>(v, tid, X);
        __syncthreads();
        if (nxt.valid && tid == 0) fetch(nxt);
        k2_phase_c<N, ACC, true, TUNE>(v, tid, X, p, row, p.tw, twr, acc);
        parity ^= 1u;
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
typedef CUresult (*tmap_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
tmap_encode_fn tmap_encoder();   // spx_stft2.cu: cuTensorMapEncodeTiled through cudaGetDriverEntryPoint (no libcuda link)

// the tensor copy addresses frames in rows of 128 bytes relative to the input pointer
inline bool stft2_ok(const StftLaunch& L) {
    const long long elt = L.in_fmt == FMT_CF32 ? 8 : 4;
    if (((uintptr_t)L.p.in & 127u) != 0) return false;
    if ((L.p.hop * elt) % 128 != 0) return false;
    if (L.p.n_streams > 1 && (L.p.stream_stride * elt) % 128 != 0) return false;
    return tmap_encoder() != nullptr;
}

template <int N, int FMT, bool ACC, int OCC, int TUNE>
int launch_stft2_inst(StftLaunch& L) {
    using C = Stft2Cfg<N, FMT>;
    auto kern = stft2_kernel<N, FMT, ACC, OCC, TUNE>;
    static int occ_cache[64] = {0};
    int dev = 0;
    SPX_CUDA(cudaGetDevice(&dev));
    int occ = occ_cache[dev & 63];
    if (occ == 0) {
        SPX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
        SPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, C::THREADS, C::SMEM));
        if (occ < 1) return spx_set_error(SPX_E_CUDA, "stft2 kernel does not fit on an SM");
        occ_cache[dev & 63] = occ;
    }
    // chunking exactly as K1: <= 256 frames per chunk, chunks never cross a stream
    const long long workers_max = (long long)L.sm_count * occ * C::FPC;
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

    const long long elt = FMT == FMT_CF32 ? 8 : 4;
    const long long last_sample = (long long)(L.p.n_streams - 1) * L.p.stream_stride + (F - 1) * L.p.hop + N;
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {32, (cuuint64_t)((last_sample * elt) / 128)};
    const cuuint64_t gstride[1] = {128};
    const cuuint32_t box[2] = {32, C::ROWS};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = tmap_encoder()(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(L.p.in), gdim, gstride, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return spx_set_error(SPX_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    kern<<<(unsigned)grid, C::THREADS, C::SMEM, L.stream>>>(L.p, tmap);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

template <int FMT, bool ACC, int R, int OCC, int TUNE>
int launch_stft2_strip_inst(StftLaunch& L) {
    constexpr int N = 4096;
    using C = Stft2Cfg<N, FMT>;
    auto kern = stft2_strip_kernel<FMT, ACC, R, OCC, TUNE>;
    static int occ_cache[64] = {0};
    int dev = 0;
    SPX_CUDA(cudaGetDevice(&dev));
    int occ = occ_cache[dev & 63];
    if (occ == 0) {
        SPX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
        SPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 256, C::SMEM));
        if (occ < 1) return spx_set_error(SPX_E_CUDA, "stft2 strip kernel does not fit on an SM");
        occ_cache[dev & 63] = occ;
    }
    // long chunks (the strip only pays inside a chunk): one chunk per worker and stream where possible, <= 256 frames
    const long long workers_max = (long long)L.sm_count * occ;
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
    long long grid = L.p.total_chunks < workers_max ? L.p.total_chunks : workers_max;
    if (grid < 1) grid = 1;
    const long long elt = FMT == FMT_CF32 ? 8 : 4;
    const long long last_sample = (long long)(L.p.n_streams - 1) * L.p.stream_stride + (F - 1) * L.p.hop + N;
    CUtensorMap tmap;
    const cuuint64_t gdim[2] = {32, (cuuint64_t)((last_sample * elt) / 128)};
    const cuuint64_t gstride[1] = {128};
    const cuuint32_t box[2] = {32, C::ROWS / R};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = tmap_encoder()(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(L.p.in), gdim, gstride, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return spx_set_error(SPX_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    kern<<<(unsigned)grid, 256, C::SMEM, L.stream>>>(L.p, tmap);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

// strip staging as the default uses it: cf32, N = 4096, hop = N/4 (the caller checks the shape)
template <int TUNE>
int launch_stft2_strip(StftLaunch& L) {
    const bool acc = L.p.welch_acc != nullptr || L.p.maxhold != nullptr;
    return acc ? launch_stft2_strip_inst<FMT_CF32, true, 4, 2, TUNE>(L) : launch_stft2_strip_inst<FMT_CF32, false, 4, 2, TUNE>(L);
}

template <int N, int OCC, int TUNE>
int launch_stft2_n(StftLaunch& L) {
    const bool acc = L.p.welch_acc != nullptr || L.p.maxhold != nullptr;
    if (L.in_fmt == FMT_CF32) {
        return acc ? launch_stft2_inst<N, FMT_CF32, true, OCC, TUNE>(L) : launch_stft2_inst<N, FMT_CF32, false, OCC, TUNE>(L);
    }
    return acc ? launch_stft2_inst<N, FMT_CI16, true, OCC, TUNE>(L) : launch_stft2_inst<N, FMT_CI16, false, OCC, TUNE>(L);
}

int launch_stft2(StftLaunch& L);   // spx_stft2.cu: N = 1024, 2048, 4096

}  // namespace spx
