// spx_detect_device.cuh -- per-cell steps of the region labelling (K11, spx_detect.cu), host and device.
//
// Labels are a parent array over the cells' raster indices i = r * cols + c: L[i] = -1 for a cell outside the mask, else a
// parent <= i, and L[i] == i for a root.  Every union links the larger of two roots below the smaller one with an atomic
// minimum, so a parent is always a smaller raster index and the root of a component is its smallest cell, whatever order
// the unions ran in.  8-connectivity: a cell links to its west, north-west, north and north-east neighbours; the pairs
// that cross a tile edge are linked again by the border pass in global memory.
//
// Kept apart from the kernels so that a CPU harness (tests/emul/detect_emul.cu) runs exactly these functions, with the
// host shims below in place of the device atomics, in any order of cells and tiles.
#pragma once
#include <stdint.h>
#include <string.h>

#define SPX_DET_HD __host__ __device__ __forceinline__

namespace spx {

constexpr int DET_TILE_H = 32, DET_TILE_W = 32;   // tile of the local pass (the harness takes other shapes)

// a parent as another thread may have just lowered it (device: volatile, so a retry reads it again)
SPX_DET_HD int det_load(const int* p) {
#ifdef __CUDA_ARCH__
    return *(const volatile int*)p;
#else
    return *p;
#endif
}

SPX_DET_HD int det_atomic_min(int* p, int v) {
#ifdef __CUDA_ARCH__
    return atomicMin(p, v);
#else
    const int o = *p;
    if (v < o) *p = v;
    return o;
#endif
}

SPX_DET_HD int det_find(const int* L, int x) {
    int p;
    while ((p = det_load(L + x)) != x) x = p;
    return x;
}

// Lock-free union (Playne & Hawick): find both roots, lower the larger toward the smaller, and retry from the old parent
// when the larger root was linked elsewhere in the meantime (its old link is then joined to the smaller root as well).
SPX_DET_HD void det_union(int* L, int a, int b) {
    for (;;) {
        a = det_find(L, a);
        b = det_find(L, b);
        if (a == b) return;
        if (a > b) { const int t = a; a = b; b = t; }
        const int old = det_atomic_min(L + b, a);
        if (old == b) return;
        b = old;
    }
}

// union of cell (r, c) with (r + dr, c + dc) of a box of h x w cells stored with row pitch `pitch`, when that neighbour is
// inside the box and in the mask
SPX_DET_HD void det_link(int* L, int r, int c, int dr, int dc, int h, int w, int pitch) {
    const int r2 = r + dr, c2 = c + dc;
    if (r2 < 0 || r2 >= h || c2 < 0 || c2 >= w) return;
    const int j = r2 * pitch + c2;
    if (det_load(L + j) < 0) return;
    det_union(L, r * pitch + c, j);
}

// The mask: float64(v) >= floor + threshold (`level`), so NaN cells and NaN floors are out, as numpy compares them.
SPX_DET_HD bool det_in_mask(float v, double level) { return (double)v >= level; }

// ---- local pass: one tile of h x w valid cells in T[th * tw], local index li = lr * tw + lc
SPX_DET_HD void det_tile_init(int* T, int li, bool in_mask) { T[li] = in_mask ? li : -1; }

// the four backward neighbours of a cell of the tile that is in the mask
SPX_DET_HD void det_tile_link(int* T, int lr, int lc, int h, int w, int tw) {
    det_link(T, lr, lc, 0, -1, h, w, tw);
    det_link(T, lr, lc, -1, -1, h, w, tw);
    det_link(T, lr, lc, -1, 0, h, w, tw);
    det_link(T, lr, lc, -1, 1, h, w, tw);
}

// global parent of a tile cell after the local unions: the raster index of its local root (-1 outside the mask).  The
// local raster order is the global one restricted to the tile, so the local root is the component's smallest cell there.
SPX_DET_HD int det_tile_parent(const int* T, int li, int r0, int c0, int tw, int cols) {
    if (det_load(T + li) < 0) return -1;
    const int root = det_find(T, li);
    return (r0 + root / tw) * cols + c0 + root % tw;
}

// ---- border pass over the global parents of a rows x cols image cut in tiles of th x tw
// a cell in the first column of a tile (c > 0): its west, north-west and south-west neighbours in the tile to the left
SPX_DET_HD void det_border_left(int* L, int r, int c, int rows, int cols) {
    det_link(L, r, c, 0, -1, rows, cols, cols);
    det_link(L, r, c, -1, -1, rows, cols, cols);
    det_link(L, r, c, 1, -1, rows, cols, cols);
}
// a cell in the first row of a tile (r > 0): its north-west, north and north-east neighbours in the tile above
SPX_DET_HD void det_border_top(int* L, int r, int c, int rows, int cols) {
    det_link(L, r, c, -1, -1, rows, cols, cols);
    det_link(L, r, c, -1, 0, rows, cols, cols);
    det_link(L, r, c, -1, 1, rows, cols, cols);
}

// ---- numbering: after the roots are numbered, a root's parent slot holds -(id + 2)
SPX_DET_HD int det_encode_id(int id) { return -(id + 2); }
// component number of cell i (-1: outside the mask)
SPX_DET_HD int det_component(const int* L, int i) {
    const int v = L[i];
    if (v == -1) return -1;
    return v < -1 ? -v - 2 : -L[v] - 2;
}

// peak key: order-preserving bits of the float32 value in the high word (-0 counted as +0, as numpy's max ties them), the
// complement of the raster index in the low word, so the 64-bit maximum is the largest value at its smallest index
SPX_DET_HD unsigned long long det_peak_key(float v, int idx) {
    const float z = v + 0.0f;
    uint32_t u;
#ifdef __CUDA_ARCH__
    u = __float_as_uint(z);
#else
    memcpy(&u, &z, 4);
#endif
    const uint32_t k = (u >> 31) ? ~u : (u | 0x80000000u);
    return ((unsigned long long)k << 32) | (unsigned long long)(~(uint32_t)idx);
}
SPX_DET_HD int det_peak_index(unsigned long long key) { return (int)~(uint32_t)(key & 0xffffffffull); }

}  // namespace spx
