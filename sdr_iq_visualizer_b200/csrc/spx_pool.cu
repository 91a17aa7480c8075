// spx_pool.cu -- pooled spectrogram: display-detector rows of K frames x B bins (DESIGN.md section 4, K8).
//
//   mean: acc[s][g][c] += sum of (10^(d/20) - eps)^2 over the cell      max: acc[s][g][c] = max(acc, max of d over the cell)
//
// for the float32 dB rows d = rows[s][f][j] of a batch whose frame 0 is global frame `frame0`; row g = (frame0 + f) / K,
// column c = j / B.  A thread owns 4 adjacent bins (one float4 per row when N % 4 == 0 and the rows are 16-byte aligned),
// a CTA a strip of 4 * blockDim bins and a chunk of frames of one stream.  The rows are read once; the thread keeps its
// partials in registers (float over POOL_UNROLL rows, then float64 for the mean) and flushes them to `acc` with atomics
// whenever a pooled row ends and at the end of its chunk.  Before the flush the partials of one cell are combined: inside
// the thread, and across the lanes that share the cell with shuffles when B % 4 == 0 and B / 4 is a power of two.
#include <math.h>
#include <stdint.h>

#include "spx_plan.h"
#include "spx_pool_device.cuh"

namespace spx {

constexpr int POOL_THREADS = 256;
constexpr int POOL_UNROLL = 4;              // rows in flight per thread
constexpr long long POOL_MIN_ROWS = 16;     // rows per chunk, at least

// float64 max through the integer order of IEEE bits: non-negative values order as signed integers, negative values in
// reverse as unsigned integers (-inf, the identity, is the largest negative pattern).  +0 stands for -0.
__device__ inline void pool_atomic_max(double* addr, double v) {
    if (v >= 0.0) atomicMax(reinterpret_cast<long long*>(addr), __double_as_longlong(v == 0.0 ? 0.0 : v));
    else atomicMin(reinterpret_cast<unsigned long long*>(addr), (unsigned long long)__double_as_longlong(v));
}

template <bool MAX>
__device__ inline double pool_comb(double a, double b) { return MAX ? fmax(a, b) : a + b; }

template <bool MAX>
__device__ inline void pool_store(double* addr, double v) {
    if (MAX) {
        if (v > -INFINITY) pool_atomic_max(addr, v);   // -inf: nothing but NaN in the cell, nothing to add
    } else {
        atomicAdd(addr, v);
    }
}

// One cell row of `acc` (row g of stream s) receives this thread's partials of bins j0 .. j0 + nb - 1.
template <bool MAX>
__device__ inline void pool_flush(double* acc_g, const double (&p)[4], int j0, int nb, int B, int lanes) {
    if (lanes) {   // all 4 bins in one cell, cells start at lane groups of `lanes` (whole warps when lanes == 32)
        double v = MAX ? -INFINITY : 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (k < nb) v = pool_comb<MAX>(v, p[k]);
        for (int o = lanes >> 1; o >= 1; o >>= 1) v = pool_comb<MAX>(v, __shfl_xor_sync(0xffffffffu, v, o));
        if (nb > 0 && (threadIdx.x & (lanes - 1)) == 0) pool_store<MAX>(acc_g + j0 / B, v);
        return;
    }
    // runs of bins in the same cell, one atomic per run (unrolled: p stays in registers)
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        if (k >= nb) break;
        const int c = pool_col_of(j0 + k, B);
        if (k > 0 && pool_col_of(j0 + k - 1, B) == c) continue;   // not the first bin of its run
        double v = p[k];
#pragma unroll
        for (int m = k + 1; m < 4; ++m)
            if (m < nb && pool_col_of(j0 + m, B) == c) v = pool_comb<MAX>(v, p[m]);
        pool_store<MAX>(acc_g + c, v);
    }
}

template <bool MAX>
__global__ void __launch_bounds__(POOL_THREADS, 4)
pool_kernel(const float* __restrict__ rows, long long rows_per_stream, long long nf, int N, int B, long long K,
            long long frame0, long long rows_per_chunk, int chunks, int vec, int lanes, float eps,
            double* __restrict__ acc, long long G) {
    const int C = N / B;
    const long long s = blockIdx.y / chunks;
    const long long c0 = (blockIdx.y % chunks) * rows_per_chunk;
    const long long c1 = c0 + rows_per_chunk < nf ? c0 + rows_per_chunk : nf;
    const int j0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int nb = N - j0 >= 4 ? 4 : (N - j0 > 0 ? N - j0 : 0);
    const float* col = rows + (size_t)(s * rows_per_stream) * N + j0;
    double* acc_s = acc + (size_t)s * G * C;
    constexpr float ID = MAX ? -INFINITY : 0.f;
    // every thread walks the same segments (they depend on the block only), so the shuffles of the flush see full warps
    for (long long a = c0; a < c1;) {
        const long long g = pool_row_of(frame0 + a, K);
        long long b = (g + 1) * K - frame0;
        if (b > c1) b = c1;
        double p[4] = {ID, ID, ID, ID};
        for (long long f = a; f < b; f += POOL_UNROLL) {
            float4 v[POOL_UNROLL];
#pragma unroll
            for (int u = 0; u < POOL_UNROLL; ++u) {
                v[u] = make_float4(ID, ID, ID, ID);
                if (f + u < b && nb > 0) {
                    const float* q = col + (size_t)(f + u) * N;
                    if (vec) {
                        v[u] = __ldcs(reinterpret_cast<const float4*>(q));   // read once: evict first
                    } else {
                        v[u].x = q[0];
                        if (nb > 1) v[u].y = q[1];
                        if (nb > 2) v[u].z = q[2];
                        if (nb > 3) v[u].w = q[3];
                    }
                }
            }
            float t[4] = {ID, ID, ID, ID};
#pragma unroll
            for (int u = 0; u < POOL_UNROLL; ++u) {
                if (f + u >= b) break;
                const float e[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    t[k] = MAX ? fmaxf(t[k], e[k]) : t[k] + pool_db_to_power(e[k], eps);
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) p[k] = pool_comb<MAX>(p[k], (double)t[k]);
        }
        pool_flush<MAX>(acc_s + (size_t)g * C, p, j0, nb, B, lanes);
        a = b;
    }
}

__global__ void pool_fill_kernel(double* acc, long long n, double v) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        acc[i] = v;
}

__global__ void pool_finalize_kernel(const double* __restrict__ acc, long long n, long long G, int C, long long K,
                                     long long F_total, int B, int max_mode, float eps, float vmin, float vmax,
                                     float* __restrict__ db_out, uint8_t* __restrict__ wf_out) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long g = (i / C) % G;
        const float db = max_mode ? pool_max_db(acc[i]) : pool_mean_db(acc[i], pool_row_frames(g, K, F_total), B, eps);
        if (db_out) db_out[i] = db;
        if (wf_out) wf_out[i] = pool_level(db, vmin, vmax);
    }
}

static unsigned elementwise_blocks(long long n) {
    const long long b = (n + 255) / 256;
    return (unsigned)(b < 4096 ? (b > 0 ? b : 1) : 4096);
}

int pool_fill_launch(double* acc, long long n, int mode, cudaStream_t st) {
    if (n <= 0) return SPX_OK;
    pool_fill_kernel<<<elementwise_blocks(n), 256, 0, st>>>(acc, n, mode == SPX_POOL_MAX ? -INFINITY : 0.0);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

int pool_finalize_launch(const spx_plan* pl, const double* acc, long long n_streams, long long G, long long F_total,
                         long long K, int B, int mode, float vmin, float vmax, float* db_out, uint8_t* wf_out,
                         cudaStream_t st) {
    const int C = pl->cfg.nfft / B;
    const long long n = n_streams * G * C;
    if (n <= 0 || (!db_out && !wf_out)) return SPX_OK;
    pool_finalize_kernel<<<elementwise_blocks(n), 256, 0, st>>>(acc, n, G, C, K, F_total, B, mode == SPX_POOL_MAX ? 1 : 0,
                                                                 pl->cfg.db_eps, vmin, vmax, db_out, wf_out);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

// Frames per chunk: enough chunks for about 2048 threads per SM (two waves of the four CTAs an SM holds), at least
// POOL_MIN_ROWS rows each.
int pool_launch(const spx_plan* pl, const float* rows, long long n_streams, long long frames, long long frame0,
                const PoolCall& pc, double* acc, cudaStream_t st) {
    if (frames <= 0 || n_streams <= 0) return SPX_OK;
    const int N = pl->cfg.nfft, B = pc.bins_per_col;
    const int threads = (N + 3) / 4 >= POOL_THREADS ? POOL_THREADS : (((N + 3) / 4 + 31) / 32) * 32;
    const long long strips = (N + 4LL * threads - 1) / (4LL * threads);
    const int vec = (N % 4 == 0 && ((uintptr_t)rows & 15u) == 0) ? 1 : 0;
    int lanes = 0;
    if (B % 4 == 0 && ((B / 4) & (B / 4 - 1)) == 0) lanes = B / 4 < 32 ? B / 4 : 32;
    const long long target = (long long)(pl->sm_count > 0 ? pl->sm_count : 148) * (2048 / threads);
    long long chunks = (target + strips * n_streams - 1) / (strips * n_streams);
    long long per = (frames + chunks - 1) / chunks;
    if (per < POOL_MIN_ROWS) per = POOL_MIN_ROWS;
    chunks = (frames + per - 1) / per;
    // gridDim.y = streams x chunks <= 65535: streams go in groups when there are more
    const long long max_y = 65535;
    if (chunks > max_y) {
        chunks = max_y;
        per = (frames + chunks - 1) / chunks;
        chunks = (frames + per - 1) / per;
    }
    const long long group = max_y / chunks < n_streams ? max_y / chunks : n_streams;
    const long long C = N / B;
    for (long long g0 = 0; g0 < n_streams; g0 += group) {
        const long long ng = n_streams - g0 < group ? n_streams - g0 : group;
        dim3 grid((unsigned)strips, (unsigned)(ng * chunks));
        const float* r = rows + (size_t)(g0 * frames) * N;
        double* a = acc + (size_t)(g0 * pc.n_rows) * C;
        if (pc.mode == SPX_POOL_MAX)
            pool_kernel<true><<<grid, threads, 0, st>>>(r, frames, frames, N, B, pc.frames_per_row, frame0, per,
                                                        (int)chunks, vec, lanes, pl->cfg.db_eps, a, pc.n_rows);
        else
            pool_kernel<false><<<grid, threads, 0, st>>>(r, frames, frames, N, B, pc.frames_per_row, frame0, per,
                                                         (int)chunks, vec, lanes, pl->cfg.db_eps, a, pc.n_rows);
        SPX_CUDA(cudaGetLastError());
    }
    return SPX_OK;
}

}  // namespace spx
