// spx_persist.cu -- persistence spectrum: per-bin histograms of the uint8 waterfall levels (DESIGN.md section 4, K7).
//
//   counts[s][q][j] = #{ f in [0, F) : rows[s*F + f][j] == q }      uint32 [S][256][N]
//
// One CTA owns a strip of PERSIST_W = 128 columns x 256 levels of uint32 counters in shared memory (128 KiB) and one
// chunk of frames of one stream.  A warp takes one row per step: lane l loads the 4 bytes of columns 4l .. 4l+3 (one
// coalesced 128-byte load per warp) and adds byte b to counter slot 32b + l of its level.  For a fixed b the 32 lanes
// then hit 32 different banks whatever their levels; neighbouring rows mostly share a level in the same column, so a
// warp never spreads one row's column over several lanes of the same instruction (those would be same-address
// atomics, which serialise).  At the end the CTA adds its non-zero counters to global memory, undoing the slot map.
#include <stdint.h>

#include "spx_plan.h"

namespace spx {

constexpr int PERSIST_W = 128;        // columns per strip
constexpr int PERSIST_THREADS = 1024;
constexpr int PERSIST_UNROLL = 4;     // rows in flight per warp
constexpr long long PERSIST_MIN_ROWS = 256;   // rows per chunk, at least: the zero + flush of a table is 64 K words

// column c (0..127) of a strip -> its counter slot in the strip's level row, and back
__host__ __device__ inline int persist_slot(int c) { return 32 * (c & 3) + (c >> 2); }
__host__ __device__ inline int persist_col(int slot) { return 4 * (slot & 31) + (slot >> 5); }

__global__ void __launch_bounds__(PERSIST_THREADS, 1)
persist_kernel(const uint8_t* __restrict__ rows, long long F, int N, long long rows_per_chunk, int chunks, int vec,
               uint32_t* __restrict__ counts) {
    extern __shared__ uint4 persist_smem[];
    uint32_t* tab = reinterpret_cast<uint32_t*>(persist_smem);   // [256 levels][PERSIST_W slots]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = PERSIST_THREADS / 32;
    const int s0 = blockIdx.x * PERSIST_W;
    const long long s = blockIdx.y / chunks;
    const long long f0 = (blockIdx.y % chunks) * rows_per_chunk;
    const long long f1 = f0 + rows_per_chunk < F ? f0 + rows_per_chunk : F;

    for (int i = tid; i < 256 * PERSIST_W / 4; i += PERSIST_THREADS) persist_smem[i] = make_uint4(0u, 0u, 0u, 0u);
    __syncthreads();

    // this lane's columns s0 + 4 lane + b, b < nb (the last strip of an N that is not a multiple of 128 is partial)
    const int c0 = s0 + 4 * lane;
    const int nb = N - c0 >= 4 ? 4 : (N - c0 > 0 ? N - c0 : 0);
    const bool word = vec && nb == 4;   // N % 4 == 0 and a 4-byte aligned base: one 32-bit load per row
    const uint8_t* col = rows + (size_t)(s * F) * N + c0;
    for (long long f = f0 + warp; f < f1; f += PERSIST_UNROLL * NW) {
        uint32_t w[PERSIST_UNROLL];
#pragma unroll
        for (int u = 0; u < PERSIST_UNROLL; ++u) {
            const long long fu = f + (long long)u * NW;
            w[u] = 0u;
            if (fu < f1 && nb > 0) {
                const uint8_t* p = col + (size_t)fu * N;
                if (word) {
                    w[u] = __ldcs(reinterpret_cast<const unsigned int*>(p));   // read once: evict first
                } else {
                    for (int b = 0; b < nb; ++b) w[u] |= (uint32_t)p[b] << (8 * b);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < PERSIST_UNROLL; ++u) {
            if (f + (long long)u * NW >= f1) break;
#pragma unroll
            for (int b = 0; b < 4; ++b)
                if (b < nb) atomicAdd(&tab[((w[u] >> (8 * b)) & 255u) * PERSIST_W + 32 * b + lane], 1u);
        }
    }
    __syncthreads();

    // flush in column order (a warp's global atomics cover 32 consecutive columns of one level)
    uint32_t* out = counts + (size_t)s * 256 * N;
    for (int i = tid; i < 256 * PERSIST_W; i += PERSIST_THREADS) {
        const int q = i / PERSIST_W, c = i % PERSIST_W;
        const uint32_t v = tab[q * PERSIST_W + persist_slot(c)];
        if (v != 0u && s0 + c < N) atomicAdd(&out[(size_t)q * N + s0 + c], v);
    }
}

// Frames per chunk: the fewest chunks whose grid fills the SMs' waves to >= 90 % (or the best fill there is), with at
// least PERSIST_MIN_ROWS rows per chunk.
static long long persist_chunks(long long units, long long F, int sm_count) {
    const long long cmax = (F + PERSIST_MIN_ROWS - 1) / PERSIST_MIN_ROWS;
    long long best = 1;
    double best_fill = 0.0;
    for (long long c = 1; c <= cmax && c <= 4096; ++c) {
        const long long ctas = units * c, waves = (ctas + sm_count - 1) / sm_count;
        const double fill = (double)ctas / (double)(waves * sm_count);
        if (fill > best_fill + 1e-9) { best = c; best_fill = fill; }
        if (fill >= 0.9) break;
    }
    return best;
}

int persist_launch(const spx_plan* pl, const uint8_t* rows, long long n_streams, long long frames, uint32_t* counts,
                   cudaStream_t st) {
    if (frames <= 0 || n_streams <= 0) return SPX_OK;
    const int N = pl->cfg.nfft;
    const int smem = 256 * PERSIST_W * (int)sizeof(uint32_t);
    SPX_TRY(kernel_setup((const void*)persist_kernel, PERSIST_THREADS, smem, nullptr));
    const long long strips = (N + PERSIST_W - 1) / PERSIST_W;
    const int vec = (N % 4 == 0 && ((uintptr_t)rows & 3u) == 0) ? 1 : 0;
    // gridDim.y = streams x chunks <= 65535: streams go in groups when there are more
    const long long max_y = 65535;
    long long chunks = persist_chunks(strips * n_streams, frames, pl->sm_count > 0 ? pl->sm_count : 148);
    if (chunks > max_y) chunks = max_y;
    const long long group = max_y / chunks < n_streams ? max_y / chunks : n_streams;
    const long long per = (frames + chunks - 1) / chunks;
    for (long long g0 = 0; g0 < n_streams; g0 += group) {
        const long long ng = n_streams - g0 < group ? n_streams - g0 : group;
        dim3 grid((unsigned)strips, (unsigned)(ng * chunks));
        persist_kernel<<<grid, PERSIST_THREADS, smem, st>>>(rows + (size_t)(g0 * frames) * N, frames, N, per, (int)chunks,
                                                           vec, counts + (size_t)g0 * 256 * N);
        SPX_CUDA(cudaGetLastError());
    }
    return SPX_OK;
}

}  // namespace spx
