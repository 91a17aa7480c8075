// spx_big2.cu -- K2v2: the 65536-point STFT (BASELINE config 5) as ONE persistent kernel (device pieces and the data
// flow are described in spx_big2_device.cuh).
//
// Grid = lanes x 16 CTAs, all co-resident (cooperative launch).  The 16 CTAs of a lane share the lane's frames
// f = lane, lane + lanes, ...: in role A CTA g transforms column tile g of a frame and writes its slice of the scratch T,
// in role B it transforms row tile g of a frame the lane produced `lag` steps earlier.  The hand-over is a per-(lane, slot)
// counter: one release-increment per producer warp (16 CTAs x 8 warps), a relaxed poll by the consumer's elected thread
// before it issues the TMA load of its row tile.  The scratch (lanes x (2 lag + 2) x 512 KiB = 54 MB at 18 lanes, lag 2)
// stays resident in the 126 MB L2: DRAM sees the capture once and the uint8 rows once (ncu: 1.08 x the algorithmic bytes).
// No block-wide barrier in role A (tile hand-over by mbarriers, warp-local exchange); one in role B (byte tile transpose).
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "spx_big2_device.cuh"
#include "spx_plan.h"
#include "spx_stft2_kernel.cuh"
#include "spx_tables.h"

namespace spx {

struct Big2Params {
    const float* wtab;       // [16 g][16 a][256 tid] window * scale in phase A's thread order, or nullptr (rect, scale 1)
    const float2* tw4096;    // N = 4096 twiddle table (its pass-1 rows are W_256^{b k_a})
    const float2* bases;     // [16 g][7][256] float2, see big2_twiddle_store
    float2* scratch;         // [lanes][slots][65536]
    int* done;               // [lanes][slots] producer counters, zeroed before the launch
    long long frames;        // frames of this launch
    long long row0;          // output row of frame 0
    unsigned char* wf_rows;
    double* welch_acc;
    float* maxhold;
    float db_eps, db_pw_min, q_a, q_b;
    int sys_atomics;
    int in_row0;             // tensor row (256 samples each) of frame 0
    int hop_rows;            // hop / 256
    int lanes;
    int lag, slots;          // slots = 2 lag + 2
    int rotate;              // duty rotation among the warps (env SPX_BIG2_ROTATE, default 1)
    int l2_prefetch;         // request the next frame's column tile into L2 one role early (on for hop >= N; env SPX_BIG2_L2PF)
};

// shared memory: [staging tile 32 KB, 1024-aligned][warp-local exchange buffer][window of this column tile, [16 a][256 tid]]
// [twiddle bases of this column tile, [7][256]][two uint8 tiles]
enum { BIG2_X_BYTES = 16 * 280 * 8, BIG2_STAGE = 32768, BIG2_WFULL = 16384, BIG2_BASES = 7 * 256 * 8, BIG2_U8 = 2 * 4096 };
enum { BIG2_SMEM = BIG2_STAGE + BIG2_X_BYTES + BIG2_WFULL + BIG2_BASES + BIG2_U8 + 1024 };
constexpr int BIG2_TUNE = TUNE_FMADFT | TUNE_QFMA;
// Lag D between producing a frame's scratch (role A) and consuming it (role B), in steps of the lane; scratch slots per
// lane = 2 D + 2: a CTA that starts A(s) has finished B(s-D-1), so all 16 CTAs of its lane have finished A(s-D-1) and
// therefore everything before it in their sequence -- including B(s-2D-2), the last reader of slot s mod (2D+2).
// D = 1: 18 lanes x 4 slots x 512 KiB = 36 MB of scratch stays in L2 (ncu: DRAM traffic 1.08 x algorithmic); with D = 2
// (54 MB) the scratch starts to spill to HBM (ncu: 813 MB written per 2^26 samples instead of 186 MB).
constexpr int BIG2_LAG_DEFAULT = 1, BIG2_LAG_MAX = 4;    // plan knob: env SPX_BIG2_LAG

__device__ __forceinline__ int ld_relaxed_gpu(const int* p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void tma_load_tile(unsigned dst, const CUtensorMap* tmap, int x, int y, unsigned bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(tmap), "r"(x), "r"(y), "r"(bar)
                 : "memory");
}

__device__ __forceinline__ void tma_prefetch_tile_l2(const CUtensorMap* tmap, int x, int y) {
    asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(tmap), "r"(x), "r"(y) : "memory");
}

// The role sequence of a CTA with lag D: iteration i runs A(i) (if i < n) and then B(i - D) (if 0 <= i - D < n).
struct Big2Seq {
    int it, ph;      // ph 0 = the A place of iteration `it`, 1 = its B place
    __device__ __forceinline__ bool valid(int n, int lag) const { return ph == 0 ? it < n : (it >= lag && it - lag < n); }
    __device__ __forceinline__ bool advance(int n, int lag) {   // to the next existing role; false at the end
        while (true) {
            if (ph == 0) ph = 1;
            else { ph = 0; ++it; }
            if (it >= n + lag) return false;
            if (valid(n, lag)) return true;
        }
    }
    __device__ __forceinline__ int s(int lag) const { return ph == 0 ? it : it - lag; }
};

template <bool ACC, int FMT>
__global__ void __launch_bounds__(256, 2)
big2_kernel(const Big2Params p, const __grid_constant__ CUtensorMap tm_in, const __grid_constant__ CUtensorMap tm_t) {
    extern __shared__ unsigned char smem_raw_b2[];
    __shared__ unsigned long long mbar;
    const int tid = threadIdx.x;
    const int lane = blockIdx.x >> 4, g = blockIdx.x & 15;
    const unsigned raw_u32 = smem_u32(smem_raw_b2);
    unsigned char* base = smem_raw_b2 + (((raw_u32 + 1023u) & ~1023u) - raw_u32);
    unsigned char* stage = base;
    float2* X = reinterpret_cast<float2*>(base + BIG2_STAGE);
    float* wfull = reinterpret_cast<float*>(base + BIG2_STAGE + BIG2_X_BYTES);
    float2* bases = reinterpret_cast<float2*>(base + BIG2_STAGE + BIG2_X_BYTES + BIG2_WFULL);
    unsigned char* u8tile = base + BIG2_STAGE + BIG2_X_BYTES + BIG2_WFULL + BIG2_BASES;
    const unsigned full_u32 = smem_u32(&mbar), stage_u32 = smem_u32(stage);

    // frames of this lane: f_s = lane + s * lanes, s in [0, n_l)
    const int n_l = p.frames > lane ? (int)((p.frames - lane + p.lanes - 1) / p.lanes) : 0;
    if (n_l == 0) return;
    const int lag = p.lag, slots = p.slots;
    if (p.wtab != nullptr)
        for (int i = tid; i < 16 * 256; i += 256) wfull[i] = __ldg(p.wtab + (size_t)g * 4096 + i);
    for (int i = tid; i < 7 * 256; i += 256) bases[i] = __ldg(p.bases + (size_t)g * 7 * 256 + i);
    if (tid == 0) mbar_init(full_u32, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    // six register bases of W_256^{b k_a} per thread, nine derived products per role: a 15 x 16 shared-memory table instead
    // (k2_phase_b1_tab) measured 5 % slower on the config-5 shape (112.6 vs 118.2 GS/s)
    TwRegs<4096> twr;
    tw_regs_load_pass<4096, 1>(twr, k2_ka_of(tid), p.tw4096);
    StftAcc<ACC> acc;
    acc.reset();
    int* const done = p.done + lane * slots;
    const float* wf_ptr = p.wtab != nullptr ? wfull + tid : nullptr;

    auto issue = [&](int kind, int s) {     // elected thread: start the TMA load of that role's tile
        if (kind == 0) {   // cf32: box {128 B, 256 rows}; ci16: box {64 B, 256 rows} (x in 4-byte units)
            mbar_expect_tx(full_u32, FMT == FMT_CF32 ? BIG2_STAGE : BIG2_STAGE / 2);
            tma_load_tile(stage_u32, &tm_in, (FMT == FMT_CF32 ? 32 : 16) * g, p.in_row0 + (lane + s * p.lanes) * p.hop_rows, full_u32);
        } else {
            mbar_expect_tx(full_u32, BIG2_STAGE);
            const int slot = s % slots;
            const int target = 16 * (s / slots + 1);       // the 16 CTAs of the lane release once per visit of the slot
            // the tile is read by the TMA unit straight from L2 (the point of coherence), never through this SM's L1: a
            // relaxed poll is enough, no L1 invalidation (an acquire load flushes L1 and the local-memory lines in it)
            while (ld_relaxed_gpu(done + slot) < target) __nanosleep(100);
            asm volatile("fence.proxy.async.global;" ::: "memory");   // generic-proxy writes of the producers -> async-proxy read
            tma_load_tile(stage_u32, &tm_t, 32 * g, (lane * slots + slot) * 256, full_u32);
        }
    };
    // Release of an A role (its scratch stores become visible device-wide before the counter moves): ONE fence per CTA and
    // role, issued by one lane after a block barrier that orders every warp's stores before it (cumulativity).  The fence
    // (MEMBAR.GPU, ~0.5 us even with no store in flight) is paid by a different warp each role.
    auto release = [&](int slot, int duty_warp) {
        if (tid == 32 * duty_warp) asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(done + slot) : "memory");
    };
    auto store_run = [&](int buf, int s_row) {   // run k2s = tid of the row of frame s_row: 16 consecutive bins 256 k2s + 16 g .. + 15
        const uint4 run = *reinterpret_cast<const uint4*>(u8tile + buf * 4096 + 16 * tid);
        const long long f = lane + (long long)s_row * p.lanes;
        __stcs(reinterpret_cast<uint4*>(p.wf_rows + (size_t)(p.row0 + f) * BIG2_N + 256 * tid + 16 * g), run);
    };

    Big2Seq cur{0, 0};
    unsigned parity = 0;           // bit 0: phase parity of the staging barrier; the role counter lives in bits 1..
    int pend_slot = -1;            // A role whose release is still owed (done one role later, behind the next block barrier)
    int pend_s = -1;               // B role (frame index s) whose uint8 tile is still to be stored (same place)
    float2 v[16];
    if (tid == 0) issue(0, 0);
    while (true) {
        const int kind = cur.ph, s = cur.s(lag);
        Big2Seq nx = cur;
        const bool has_next = nx.advance(n_l, lag);
        // the next role is the B role of the very frame this A role produces (a lane with a single frame): its tile can only
        // be requested after this role's release
        const bool hold = has_next && kind == 0 && nx.ph == 1 && nx.s(lag) == s;
        // the column tile of this lane's next frame comes from HBM and is only requested one role from now: ask L2 for it now
        if (p.l2_prefetch && tid == 0 && kind == 0 && s + 1 < n_l)
            tma_prefetch_tile_l2(&tm_in, (FMT == FMT_CF32 ? 32 : 16) * g, p.in_row0 + (lane + (s + 1) * p.lanes) * p.hop_rows);
        mbar_wait(full_u32, parity & 1u);
        parity += 1u;
        if (FMT == FMT_CI16 && kind == 0) big2_load_tile_ci16(v, tid, stage, wf_ptr);
        else big2_load_tile(v, tid, stage, kind == 0 ? wf_ptr : nullptr);
        // The only block barrier of the role, placed where the warps are still aligned (they all woke on the same TMA
        // completion): the staged tile is consumed (every value went through a butterfly above), the previous role's scratch
        // stores are issued and its uint8 tile is complete.  The exchange through X below is warp-local (__syncwarp).
        __syncthreads();
        const int duty = (p.rotate ? (int)(parity >> 1) : 0) & 7;     // the warp that pays for this role's fence / poll
        if (pend_slot >= 0) {
            release(pend_slot, duty);
            pend_slot = -1;
        }
        if (pend_s >= 0) {
            store_run(pend_s & 1, pend_s);
            pend_s = -1;
        }
        if (tid == 0 && has_next && !hold) issue(nx.ph, nx.s(lag));   // refill the staging tile: overlaps the whole transform
        big2_dft_store(v, tid, X);
        __syncwarp();
        k2_phase_b1<4096, BIG2_TUNE>(v, tid, X, twr);
        if (kind == 0) {
            const int slot = s % slots;
            float2* t_tile = p.scratch + ((size_t)(lane * slots + slot) << 16) + (size_t)g * 4096;
            big2_twiddle_store<BIG2_TUNE>(v, tid, bases, t_tile);
            pend_slot = slot;
            if (hold) {
                __syncthreads();
                release(slot, 0);
                pend_slot = -1;
                if (tid == 0) issue(nx.ph, nx.s(lag));
            }
        } else {
            big2_epilogue<ACC, BIG2_TUNE>(v, tid, p.db_eps, p.db_pw_min, p.q_a, p.q_b, p.wf_rows != nullptr, acc, u8tile + (s & 1) * 4096);
            if (p.wf_rows != nullptr) pend_s = s;
            if (ACC) {
                if ((s & 255) == 255 || s + 1 == n_l) {   // bound the float32 accumulation like K1's chunks
#pragma unroll
                    for (int kb = 0; kb < 16; ++kb)
                        flush_acc(p.welch_acc, p.maxhold, big2_acc_pos(g, tid, kb), acc.sum[kb], acc.mx[kb], p.sys_atomics);
                    acc.reset();
                }
            }
        }
        if (!has_next) break;
        cur = nx;
    }
    if (pend_s >= 0) {
        __syncthreads();
        store_run(pend_s & 1, pend_s);
    }
}

// ------------------------------------------------------------------ host side
int big2_plan_init(spx_plan* pl) {
    if (pl->cfg.nfft != BIG2_N) return SPX_OK;
    std::vector<float2> tw = build_twiddles(4096);
    std::vector<float2> bases((size_t)16 * 7 * 256);
    const double two_pi = 6.283185307179586476925286766559;
    for (int g = 0; g < 16; ++g)
        for (int tid = 0; tid < 256; ++tid) {
            unsigned e[7];
            big2_base_exponents(g, tid, e);
            for (int q = 0; q < 7; ++q) {
                const double a = -two_pi * (double)e[q] / (double)BIG2_N;
                bases[((size_t)g * 7 + q) * 256 + tid] = make_float2((float)cos(a), (float)sin(a));
            }
        }
    SPX_CUDA(cudaMalloc(&pl->d_big2, (tw.size() + bases.size()) * sizeof(float2)));
    SPX_CUDA(cudaMemcpy(pl->d_big2, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice));
    SPX_CUDA(cudaMemcpy(pl->d_big2 + tw.size(), bases.data(), bases.size() * sizeof(float2), cudaMemcpyHostToDevice));
    pl->big2_tw_count = tw.size();
    if (pl->cfg.window != SPX_WINDOW_RECT || pl->cfg.in_scale != 1.0f) {
        // window * scale (float64 as numpy builds it, rounded once) in phase A's thread order: [16 g][16 a][256 tid]
        std::vector<float> wt((size_t)16 * 16 * 256);
        for (int g = 0; g < 16; ++g)
            for (int a = 0; a < 16; ++a)
                for (int tid = 0; tid < 256; ++tid)
                    wt[((size_t)g * 16 + a) * 256 + tid] = (float)(pl->win64[(size_t)big2_sample_of(g, a, tid)] * (double)pl->cfg.in_scale);
        SPX_CUDA(cudaMalloc(&pl->d_big2_win, wt.size() * sizeof(float)));
        SPX_CUDA(cudaMemcpy(pl->d_big2_win, wt.data(), wt.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    return SPX_OK;
}

// K2v2 handles: cf32 or ci16 input, N = 65536, hop a multiple of 256 samples, 16-byte aligned stream start, outputs among
// {uint8 rows, Welch sum, max-hold}.  Everything else goes through the two-kernel path of spx_bigfft.cu.
bool big2_eligible(const spx_plan* pl, const void* in, const StftOut& out) {
    if (pl->cfg.nfft != BIG2_N || pl->d_big2 == nullptr) return false;
    if (pl->cfg.variant == 1) return false;                    // variant 1 = the round-1 two-kernel path, kept for comparison
    if (out.db != nullptr || out.spec != nullptr) return false;
    if (pl->cfg.hop % 256 != 0 || ((uintptr_t)in & 15u) != 0) return false;
    return tmap_encoder() != nullptr;
}

int big2_launch_stream(spx_plan* pl, const void* in, long long frames, long long row0, const StftOut& out, cudaStream_t st) {
    if (frames <= 0) return SPX_OK;
    const bool acc = out.welch != nullptr || out.maxhold != nullptr;
    const bool ci16 = pl->cfg.in_fmt == SPX_FMT_CI16;
    auto k_acc = ci16 ? big2_kernel<true, FMT_CI16> : big2_kernel<true, FMT_CF32>;
    auto k_rows = ci16 ? big2_kernel<false, FMT_CI16> : big2_kernel<false, FMT_CF32>;
    int o1 = 0, o2 = 0;
    SPX_TRY(kernel_setup((const void*)k_acc, 256, BIG2_SMEM, &o1));
    SPX_TRY(kernel_setup((const void*)k_rows, 256, BIG2_SMEM, &o2));
    const int o = o1 < o2 ? o1 : o2;
    if (o < 1) return spx_set_error(SPX_E_CUDA, "big2 kernel does not fit on an SM");
    long long lanes = (long long)pl->sm_count * o / 16;
    if (lanes < 1) return spx_set_error(SPX_E_CUDA, "big2 kernel: fewer than 16 resident CTAs");
    if (lanes > frames) lanes = frames;
    int lag = BIG2_LAG_DEFAULT;
    if (const char* e = getenv("SPX_BIG2_LAG")) lag = atoi(e);
    if (lag < 1) lag = 1;
    if (lag > BIG2_LAG_MAX) lag = BIG2_LAG_MAX;
    const int slots = 2 * lag + 2;
    const size_t scratch_bytes = (size_t)lanes * slots * BIG2_N * sizeof(float2);
    SPX_TRY(pl->st_big.reserve(scratch_bytes + 4096));
    Big2Params p;
    memset(&p, 0, sizeof(p));
    p.wtab = pl->d_big2_win;
    p.tw4096 = pl->d_big2;
    p.bases = pl->d_big2 + pl->big2_tw_count;
    p.scratch = (float2*)pl->st_big.ptr;
    p.done = (int*)((char*)pl->st_big.ptr + scratch_bytes);
    p.frames = frames;
    p.row0 = row0;
    p.wf_rows = out.wf;
    p.welch_acc = out.welch;
    p.maxhold = out.maxhold;
    p.db_eps = pl->cfg.db_eps;
    p.db_pw_min = db_pw_min(pl);
    p.q_a = out.q_a();
    p.q_b = out.q_b();
    p.sys_atomics = out.sys_atomics;
    p.in_row0 = 0;
    p.hop_rows = pl->cfg.hop / 256;
    p.lanes = (int)lanes;
    p.lag = lag;
    p.rotate = 1;
    if (const char* e = getenv("SPX_BIG2_ROTATE")) p.rotate = atoi(e);
    // measured (profiles/r02_k2v2_l2_prefetch_ab.txt): + 2 % without overlap (hop = N: the whole tile comes from HBM), - 1 % at 50 %
    // overlap (half of the tile is an L2 hit already)
    p.l2_prefetch = p.hop_rows >= 256 ? 1 : 0;
    if (const char* e = getenv("SPX_BIG2_L2PF")) p.l2_prefetch = atoi(e);
    p.slots = slots;
    SPX_CUDA(cudaMemsetAsync(p.done, 0, (size_t)lanes * slots * sizeof(int), st));

    CUtensorMap tm_in, tm_t;
    const cuuint64_t gstride[1] = {2048};
    const cuuint32_t box[2] = {32, 256}, estr[2] = {1, 1};
    const cuuint64_t gdim_in[2] = {512, (cuuint64_t)(((frames - 1) * (long long)pl->cfg.hop + BIG2_N) / 256)};
    const cuuint64_t gdim_t[2] = {512, (cuuint64_t)(lanes * slots * 256)};
    CUresult r;
    if (ci16) {   // rows of 256 samples = 1 KB, column tile = 16 samples = 64 B
        const cuuint64_t gstride_i[1] = {1024}, gdim_i[2] = {256, gdim_in[1]};
        const cuuint32_t box_i[2] = {16, 256};
        r = tmap_encoder()(&tm_in, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(in), gdim_i, gstride_i, box_i, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    } else {
        r = tmap_encoder()(&tm_in, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(in), gdim_in, gstride, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    }
    if (r == CUDA_SUCCESS)
        r = tmap_encoder()(&tm_t, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, p.scratch, gdim_t, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return spx_set_error(SPX_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    void* args[3] = {&p, &tm_in, &tm_t};
    // cooperative launch: every CTA spins on counters written by other CTAs, so all of them must be co-resident
    SPX_CUDA(cudaLaunchCooperativeKernel(acc ? (const void*)k_acc : (const void*)k_rows, dim3((unsigned)(lanes * 16)), dim3(256), args,
                                         BIG2_SMEM, st));
    return SPX_OK;
}

}  // namespace spx
