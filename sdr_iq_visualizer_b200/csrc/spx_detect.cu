// spx_detect.cu -- K11: regions of a dB image above each row's noise floor, labelled on the GPU (spx_detect_regions).
//
// Passes, all on one stream:
//   K3        row floors: features_kernel<float> over the image rows (np.percentile(row, 20), NaN rules included)
//   local     one CTA per 32 x 32 tile: mask against the row floors, union-find in shared memory, global parents
//   border    unions across tile edges and corners in global memory (atomicMin of the larger root)
//   flatten   every cell's parent becomes its root, the component's smallest raster index; roots counted per chunk
//   scan      exclusive scan of the chunk counts: roots numbered in raster order (scipy.ndimage.label's numbering)
//   assign    each root's slot takes its number; its statistics are reset
//   stats     per cell, warp-aggregated atomics: count, bounding box, peak key, power sum
//   keep      components with >= min_cells cells counted per chunk, scanned again: the numbering after the filter
//   number    the region table, and the new number of every component
//   relabel   the label image (optional)
// The per-device staging of the plan-less calls (DeviceCtx::stage) holds the parents, the counts and the statistics.
#include <float.h>
#include <limits.h>
#include <math.h>

#include <mutex>

#include "spx_detect_device.cuh"
#include "spx_internal.h"
#include "spx_plan.h"

namespace spx {

constexpr int DET_THREADS = 256;
constexpr int DET_ITEMS = 16;                          // consecutive items per thread in the chunked passes
constexpr int DET_CHUNK = DET_THREADS * DET_ITEMS;     // items per CTA of the chunked passes
constexpr int DET_SCAN_THREADS = 1024;

// per-component statistics, structure of arrays over the component numbers
struct DetStats {
    int* n;                       // cells
    int *row0, *row1, *col0, *col1;
    unsigned long long* key;      // det_peak_key maximum
    double* power;                // sum of 10^(dB/10)
    int* new_id;                  // number after the min_cells filter, -1 if dropped
};

// exclusive scan of one value per thread over the CTA (blockDim.x a multiple of 32); every thread gets the CTA's sum
__device__ int block_excl_scan(int v, int& total) {
    __shared__ int warp_tot[DET_SCAN_THREADS / 32 + 1];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();   // warp_tot may still be read by a previous call
    if (lane == 31) warp_tot[w] = incl;
    __syncthreads();
    if (w == 0) {
        const int x = lane < nw ? warp_tot[lane] : 0;
        int xi = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, xi, o);
            if (lane >= o) xi += t;
        }
        if (lane < nw) warp_tot[lane] = xi - x;
        if (lane == nw - 1) warp_tot[DET_SCAN_THREADS / 32] = xi;
    }
    __syncthreads();
    total = warp_tot[DET_SCAN_THREADS / 32];
    return warp_tot[w] + incl - v;
}

__global__ void __launch_bounds__(DET_THREADS)
det_local_kernel(const float* __restrict__ db, long long stride, int rows, int cols, const spx_features* __restrict__ feats,
                 double thr, int* __restrict__ L) {
    __shared__ int T[DET_TILE_H * DET_TILE_W];
    __shared__ double level[DET_TILE_H];
    const int r0 = blockIdx.y * DET_TILE_H, c0 = blockIdx.x * DET_TILE_W;
    const int h = min(DET_TILE_H, rows - r0), w = min(DET_TILE_W, cols - c0);
    if ((int)threadIdx.x < h) level[threadIdx.x] = __dadd_rn(feats[r0 + threadIdx.x].noise_floor_db, thr);
    __syncthreads();
    for (int li = threadIdx.x; li < DET_TILE_H * DET_TILE_W; li += DET_THREADS) {
        const int lr = li / DET_TILE_W, lc = li % DET_TILE_W;
        const bool in = lr < h && lc < w && det_in_mask(db[(long long)(r0 + lr) * stride + c0 + lc], level[lr]);
        det_tile_init(T, li, in);
    }
    __syncthreads();
    for (int li = threadIdx.x; li < DET_TILE_H * DET_TILE_W; li += DET_THREADS)
        if (T[li] >= 0) det_tile_link(T, li / DET_TILE_W, li % DET_TILE_W, h, w, DET_TILE_W);
    __syncthreads();
    for (int li = threadIdx.x; li < DET_TILE_H * DET_TILE_W; li += DET_THREADS) {
        const int lr = li / DET_TILE_W, lc = li % DET_TILE_W;
        if (lr < h && lc < w) L[(r0 + lr) * cols + c0 + lc] = det_tile_parent(T, li, r0, c0, DET_TILE_W, cols);
    }
}

// one thread per (tile, edge cell): k < 32 the tile's first column, else its first row
__global__ void __launch_bounds__(DET_THREADS)
det_border_kernel(int* L, int rows, int cols, int tiles_x, long long n_items) {
    const long long i = blockIdx.x * (long long)DET_THREADS + threadIdx.x;
    if (i >= n_items) return;
    const int tile = (int)(i / (DET_TILE_H + DET_TILE_W)), k = (int)(i % (DET_TILE_H + DET_TILE_W));
    const int r0 = (tile / tiles_x) * DET_TILE_H, c0 = (tile % tiles_x) * DET_TILE_W;
    if (k < DET_TILE_H) {
        const int r = r0 + k;
        if (c0 > 0 && r < rows && L[r * cols + c0] >= 0) det_border_left(L, r, c0, rows, cols);
    } else {
        const int c = c0 + k - DET_TILE_H;
        if (r0 > 0 && c < cols && L[r0 * cols + c] >= 0) det_border_top(L, r0, c, rows, cols);
    }
}

// parents -> roots; counts[b] = roots among items [b CHUNK, (b + 1) CHUNK)
__global__ void __launch_bounds__(DET_THREADS) det_flatten_kernel(int* L, int n, int* __restrict__ counts) {
    const long long base = blockIdx.x * (long long)DET_CHUNK + threadIdx.x * DET_ITEMS;
    int cnt = 0;
    for (int q = 0; q < DET_ITEMS; ++q) {
        const long long i = base + q;
        if (i >= n || L[i] < 0) continue;
        const int root = det_find(L, (int)i);
        L[i] = root;
        cnt += root == i;
    }
    int total;
    block_excl_scan(cnt, total);
    if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

// in place: counts[b] -> sum of counts[0 .. b - 1]; *total = sum of all (one CTA)
__global__ void __launch_bounds__(DET_SCAN_THREADS) det_scan_kernel(int* counts, int nb, int* total) {
    const int per = (nb + DET_SCAN_THREADS - 1) / DET_SCAN_THREADS;
    const int lo = threadIdx.x * per, hi = min(nb, lo + per);
    int s = 0;
    for (int b = lo; b < hi; ++b) s += counts[b];
    int tot;
    int run = block_excl_scan(s, tot);
    for (int b = lo; b < hi; ++b) {
        const int c = counts[b];
        counts[b] = run;
        run += c;
    }
    if (threadIdx.x == 0) *total = tot;
}

// roots numbered in raster order; each root's slot takes -(id + 2) and its statistics are reset
__global__ void __launch_bounds__(DET_THREADS) det_assign_kernel(int* L, int n, const int* __restrict__ offsets, DetStats s) {
    const long long base = blockIdx.x * (long long)DET_CHUNK + threadIdx.x * DET_ITEMS;
    int cnt = 0;
    for (int q = 0; q < DET_ITEMS; ++q) {
        const long long i = base + q;
        cnt += i < n && L[i] == i;
    }
    int total;
    int id = offsets[blockIdx.x] + block_excl_scan(cnt, total);
    for (int q = 0; q < DET_ITEMS && cnt; ++q) {
        const long long i = base + q;
        if (i >= n || L[i] != i) continue;
        L[i] = det_encode_id(id);
        s.n[id] = 0;
        s.row0[id] = INT_MAX; s.col0[id] = INT_MAX;
        s.row1[id] = -1; s.col1[id] = -1;
        s.key[id] = 0ull;
        s.power[id] = 0.0;
        ++id;
        --cnt;
    }
}

// per cell: warp-aggregated atomics into its component's statistics (one leader per distinct component in the warp)
__global__ void __launch_bounds__(DET_THREADS)
det_stats_kernel(const float* __restrict__ db, long long stride, int cols, int n, const int* __restrict__ L, DetStats s) {
    const long long i = blockIdx.x * (long long)DET_THREADS + threadIdx.x;
    int id = -1, r = 0, c = 0;
    float v = 0.f;
    if (i < n) {
        id = det_component(L, (int)i);
        r = (int)i / cols;
        c = (int)i - r * cols;
        if (id >= 0) v = db[(long long)r * stride + c];
    }
    const int lane = threadIdx.x & 31;
    unsigned todo = __ballot_sync(0xffffffffu, id >= 0);
    while (todo) {
        const int leader = __ffs(todo) - 1;
        const int lid = __shfl_sync(0xffffffffu, id, leader);
        const bool mine = id == lid;
        int cnt = mine, rmin = mine ? r : INT_MAX, rmax = mine ? r : -1, cmin = mine ? c : INT_MAX, cmax = mine ? c : -1;
        unsigned long long key = mine ? det_peak_key(v, (int)i) : 0ull;
        double pw = mine ? exp10((double)v / 10.0) : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            rmin = min(rmin, __shfl_xor_sync(0xffffffffu, rmin, o));
            rmax = max(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
            cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
            cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
            const unsigned long long k2 = __shfl_xor_sync(0xffffffffu, key, o);
            key = k2 > key ? k2 : key;
            pw += __shfl_xor_sync(0xffffffffu, pw, o);
        }
        if (lane == leader) {
            atomicAdd(s.n + lid, cnt);
            atomicMin(s.row0 + lid, rmin);
            atomicMax(s.row1 + lid, rmax);
            atomicMin(s.col0 + lid, cmin);
            atomicMax(s.col1 + lid, cmax);
            atomicMax(s.key + lid, key);
            atomicAdd(s.power + lid, pw);
        }
        todo &= ~__ballot_sync(0xffffffffu, mine);
    }
}

// counts[b] = components with >= min_cells cells among numbers [b CHUNK, (b + 1) CHUNK) below *n_comp
__global__ void __launch_bounds__(DET_THREADS)
det_keep_kernel(const int* __restrict__ n_comp, int min_cells, DetStats s, int* __restrict__ counts) {
    const int nc = *n_comp;
    if (blockIdx.x * DET_CHUNK >= nc) {
        if (threadIdx.x == 0) counts[blockIdx.x] = 0;
        return;
    }
    const int base = blockIdx.x * DET_CHUNK + threadIdx.x * DET_ITEMS;
    int cnt = 0;
    for (int q = 0; q < DET_ITEMS; ++q) {
        const int k = base + q;
        cnt += k < nc && s.n[k] >= min_cells;
    }
    int total;
    block_excl_scan(cnt, total);
    if (threadIdx.x == 0) counts[blockIdx.x] = total;
}

// the kept components renumbered in order; the first max_regions of them written to the region table
__global__ void __launch_bounds__(DET_THREADS)
det_number_kernel(const int* __restrict__ n_comp, int min_cells, const int* __restrict__ offsets, DetStats s,
                  const float* __restrict__ db, long long stride, int cols, const spx_features* __restrict__ feats,
                  spx_region* __restrict__ out, int max_regions) {
    const int nc = *n_comp;
    if (blockIdx.x * DET_CHUNK >= nc) return;
    const int base = blockIdx.x * DET_CHUNK + threadIdx.x * DET_ITEMS;
    int cnt = 0;
    for (int q = 0; q < DET_ITEMS; ++q) {
        const int k = base + q;
        cnt += k < nc && s.n[k] >= min_cells;
    }
    int total;
    int id = offsets[blockIdx.x] + block_excl_scan(cnt, total);
    for (int q = 0; q < DET_ITEMS; ++q) {
        const int k = base + q;
        if (k >= nc) break;
        if (s.n[k] < min_cells) {
            s.new_id[k] = -1;
            continue;
        }
        s.new_id[k] = id;
        if (id < max_regions) {
            const int p = det_peak_index(s.key[k]);
            const int pr = p / cols, pc = p - pr * cols;
            spx_region g;
            g.row0 = s.row0[k]; g.row1 = s.row1[k];
            g.col0 = s.col0[k]; g.col1 = s.col1[k];
            g.n_cells = s.n[k];
            g.peak_row = pr; g.peak_col = pc;
            g.peak_db = (double)db[(long long)pr * stride + pc];
            g.peak_floor_db = feats[pr].noise_floor_db;
            g.power_sum = s.power[k];
            out[id] = g;
        }
        ++id;
    }
}

__global__ void __launch_bounds__(DET_THREADS)
det_relabel_kernel(const int* __restrict__ L, int n, const int* __restrict__ new_id, int* __restrict__ labels) {
    const long long i = blockIdx.x * (long long)DET_THREADS + threadIdx.x;
    if (i >= n) return;
    const int k = det_component(L, (int)i);
    labels[i] = k < 0 ? 0 : new_id[k] + 1;
}

static unsigned blocks_of(long long items, long long per) { return (unsigned)((items + per - 1) / per); }

}  // namespace spx

using namespace spx;

extern "C" int spx_detect_regions(int32_t device, int32_t mem, const float* db, int32_t rows, int32_t cols, int64_t stride,
                                  double threshold_db, int32_t min_cells, spx_region* regions, int32_t max_regions,
                                  int32_t* n_regions_out, int32_t* labels, double* row_floor_db, void* stream) {
    if (!n_regions_out) return spx_set_error(SPX_E_INVALID, "n_regions_out is NULL");
    if (!db) return spx_set_error(SPX_E_INVALID, "db is NULL");
    if (mem != SPX_MEM_HOST && mem != SPX_MEM_DEVICE) return spx_set_error(SPX_E_INVALID, "unknown mem %d", mem);
    if (rows < 0 || cols < 0) return spx_set_error(SPX_E_INVALID, "negative size %d x %d", rows, cols);
    if ((long long)rows * cols > INT_MAX) return spx_set_error(SPX_E_INVALID, "rows * cols = %lld > INT32_MAX", (long long)rows * cols);
    if (stride < cols) return spx_set_error(SPX_E_INVALID, "stride %lld < cols %d", (long long)stride, cols);
    if (min_cells < 1) return spx_set_error(SPX_E_INVALID, "min_cells %d < 1", min_cells);
    if (max_regions < 0) return spx_set_error(SPX_E_INVALID, "max_regions %d < 0", max_regions);
    if (!regions && max_regions > 0) return spx_set_error(SPX_E_INVALID, "regions is NULL with max_regions %d", max_regions);
    *n_regions_out = 0;
    DeviceCtx* ctx;
    SPX_TRY(device_ctx(device, &ctx));
    if (rows == 0 || cols == 0) return SPX_OK;
    std::lock_guard<std::mutex> g(ctx->mu);
    cudaStream_t st = (mem == SPX_MEM_DEVICE && stream) ? (cudaStream_t)stream : ctx->st;

    const int n = rows * cols;
    const int n_bound = ((rows + 1) / 2) * ((cols + 1) / 2);   // most 8-connected components a rows x cols mask can hold
    const int nb_cells = (int)blocks_of(n, DET_CHUNK), nb_comp = (int)blocks_of(n_bound, DET_CHUNK);
    const int table = max_regions < n_bound ? max_regions : n_bound;
    const size_t in_bytes = mem == SPX_MEM_HOST ? ((size_t)(rows - 1) * (size_t)stride + (size_t)cols) * sizeof(float) : 0;
    const size_t cb = (size_t)n_bound;
    void* part[14];
    SPX_TRY(ctx->carve({in_bytes, sizeof(spx_features) * (size_t)rows, sizeof(int) * (size_t)n, sizeof(int) * (size_t)nb_cells,
                        sizeof(int) * (size_t)nb_comp, 2 * sizeof(int), 4 * cb, 4 * cb, 4 * cb, 4 * cb, 4 * cb, 8 * cb,
                        8 * cb + 4 * cb, sizeof(spx_region) * (size_t)table + (mem == SPX_MEM_HOST && labels ? 4 * (size_t)n : 0)},
                       part));
    const float* d_db = db;
    if (mem == SPX_MEM_HOST) {
        SPX_CUDA(cudaMemcpyAsync(part[0], db, in_bytes, cudaMemcpyHostToDevice, st));
        d_db = (const float*)part[0];
    }
    spx_features* feats = (spx_features*)part[1];
    int* L = (int*)part[2];
    int* cnt_cells = (int*)part[3];
    int* cnt_comp = (int*)part[4];
    int* totals = (int*)part[5];   // [0] components, [1] regions
    DetStats s;
    s.n = (int*)part[6];
    s.row0 = (int*)part[7]; s.row1 = (int*)part[8];
    s.col0 = (int*)part[9]; s.col1 = (int*)part[10];
    s.key = (unsigned long long*)part[11];
    s.power = (double*)part[12];
    s.new_id = (int*)(s.power + cb);
    spx_region* d_regions = (spx_region*)part[13];
    int* d_labels = labels ? (mem == SPX_MEM_HOST ? (int*)(d_regions + table) : labels) : nullptr;

    // row floors: K3 over the image rows (float32, no peak list)
    SPX_TRY(features_launch(d_db, 0, cols, rows, stride, feats, nullptr, 0, nullptr, st));
    SPX_TRY(kernel_setup((const void*)det_local_kernel, DET_THREADS, 0, nullptr));
    SPX_TRY(kernel_setup((const void*)det_border_kernel, DET_THREADS, 0, nullptr));
    SPX_TRY(kernel_setup((const void*)det_flatten_kernel, DET_THREADS, 0, nullptr));
    SPX_TRY(kernel_setup((const void*)det_scan_kernel, DET_SCAN_THREADS, 0, nullptr));
    SPX_TRY(kernel_setup((const void*)det_assign_kernel, DET_THREADS, 0, nullptr));
    SPX_TRY(kernel_setup((const void*)det_stats_kernel, DET_THREADS, 0, nullptr));
    SPX_TRY(kernel_setup((const void*)det_keep_kernel, DET_THREADS, 0, nullptr));
    SPX_TRY(kernel_setup((const void*)det_number_kernel, DET_THREADS, 0, nullptr));
    SPX_TRY(kernel_setup((const void*)det_relabel_kernel, DET_THREADS, 0, nullptr));
    const int tiles_x = (int)blocks_of(cols, DET_TILE_W), tiles_y = (int)blocks_of(rows, DET_TILE_H);
    det_local_kernel<<<dim3(tiles_x, tiles_y), DET_THREADS, 0, st>>>(d_db, stride, rows, cols, feats, threshold_db, L);
    SPX_CUDA(cudaGetLastError());
    const long long n_edge = (long long)tiles_x * tiles_y * (DET_TILE_H + DET_TILE_W);
    if (tiles_x * tiles_y > 1) det_border_kernel<<<blocks_of(n_edge, DET_THREADS), DET_THREADS, 0, st>>>(L, rows, cols, tiles_x, n_edge);
    det_flatten_kernel<<<nb_cells, DET_THREADS, 0, st>>>(L, n, cnt_cells);
    det_scan_kernel<<<1, DET_SCAN_THREADS, 0, st>>>(cnt_cells, nb_cells, totals);
    det_assign_kernel<<<nb_cells, DET_THREADS, 0, st>>>(L, n, cnt_cells, s);
    det_stats_kernel<<<blocks_of(n, DET_THREADS), DET_THREADS, 0, st>>>(d_db, stride, cols, n, L, s);
    det_keep_kernel<<<nb_comp, DET_THREADS, 0, st>>>(totals, min_cells, s, cnt_comp);
    det_scan_kernel<<<1, DET_SCAN_THREADS, 0, st>>>(cnt_comp, nb_comp, totals + 1);
    det_number_kernel<<<nb_comp, DET_THREADS, 0, st>>>(totals, min_cells, cnt_comp, s, d_db, stride, cols, feats, d_regions, table);
    if (d_labels) det_relabel_kernel<<<blocks_of(n, DET_THREADS), DET_THREADS, 0, st>>>(L, n, s.new_id, d_labels);
    SPX_CUDA(cudaGetLastError());

    const cudaMemcpyKind back = mem == SPX_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    if (row_floor_db)
        SPX_CUDA(cudaMemcpy2DAsync(row_floor_db, sizeof(double), &feats->noise_floor_db, sizeof(spx_features), sizeof(double),
                                   (size_t)rows, back, st));
    if (labels && mem == SPX_MEM_HOST)
        SPX_CUDA(cudaMemcpyAsync(labels, d_labels, sizeof(int) * (size_t)n, cudaMemcpyDeviceToHost, st));
    int total = 0;
    SPX_CUDA(cudaMemcpyAsync(&total, totals + 1, sizeof(int), cudaMemcpyDeviceToHost, st));
    SPX_CUDA(cudaStreamSynchronize(st));
    const int stored = total < table ? total : table;
    if (stored > 0) {
        SPX_CUDA(cudaMemcpyAsync(regions, d_regions, sizeof(spx_region) * (size_t)stored, cudaMemcpyDeviceToHost, st));
        SPX_CUDA(cudaStreamSynchronize(st));
    }
    *n_regions_out = total;
    return SPX_OK;
}
