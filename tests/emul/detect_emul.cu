// CPU harness of the region labelling (csrc/spx_detect_device.cuh): K11's local pass, border pass, flattening and
// numbering, run on the host with the header's atomic shims, in a seeded random order of tiles and cells at every pass, so
// that tests/test_detect_cpu.py can hold the labels to scipy.ndimage.label whatever order the unions ran in.
#include <stdint.h>

#include <algorithm>
#include <random>
#include <vector>

#include "../../sdr_iq_visualizer_b200/csrc/spx_detect_device.cuh"

extern "C" {

// mask uint8 [rows][cols]; tiles of th x tw; labels_out int32 [rows][cols] (component number + 1, 0 outside the mask).
// Returns the number of components.
int emul_label(const uint8_t* mask, int rows, int cols, int th, int tw, unsigned long long seed, int* labels_out) {
    if (rows <= 0 || cols <= 0) return 0;
    std::mt19937_64 rng(seed);
    const int tiles_y = (rows + th - 1) / th, tiles_x = (cols + tw - 1) / tw, n_tiles = tiles_x * tiles_y;
    std::vector<std::vector<int>> T((size_t)n_tiles, std::vector<int>((size_t)th * tw));
    auto tile_box = [&](int t, int* r0, int* c0, int* h, int* w) {
        *r0 = (t / tiles_x) * th;
        *c0 = (t % tiles_x) * tw;
        *h = std::min(th, rows - *r0);
        *w = std::min(tw, cols - *c0);
    };
    // local pass: every tile's mask, then the unions of all tiles' cells interleaved in one random order
    std::vector<std::pair<int, int>> ops;   // (tile, local index)
    for (int t = 0; t < n_tiles; ++t) {
        int r0, c0, h, w;
        tile_box(t, &r0, &c0, &h, &w);
        for (int li = 0; li < th * tw; ++li) {
            const int lr = li / tw, lc = li % tw;
            const bool in = lr < h && lc < w && mask[(size_t)(r0 + lr) * cols + c0 + lc];
            spx::det_tile_init(T[(size_t)t].data(), li, in);
            if (in) ops.push_back({t, li});
        }
    }
    std::shuffle(ops.begin(), ops.end(), rng);
    for (const auto& op : ops) {
        int r0, c0, h, w;
        tile_box(op.first, &r0, &c0, &h, &w);
        spx::det_tile_link(T[(size_t)op.first].data(), op.second / tw, op.second % tw, h, w, tw);
    }
    std::vector<int> L((size_t)rows * cols, -1);
    std::vector<int> order((size_t)n_tiles);
    for (int t = 0; t < n_tiles; ++t) order[(size_t)t] = t;
    std::shuffle(order.begin(), order.end(), rng);
    for (int t : order) {
        int r0, c0, h, w;
        tile_box(t, &r0, &c0, &h, &w);
        for (int lr = 0; lr < h; ++lr)
            for (int lc = 0; lc < w; ++lc)
                L[(size_t)(r0 + lr) * cols + c0 + lc] = spx::det_tile_parent(T[(size_t)t].data(), lr * tw + lc, r0, c0, tw, cols);
    }
    // border pass: the first column and the first row of every tile, in one random order
    std::vector<std::pair<int, int>> edge;   // (raster index, 0 left / 1 top)
    for (int t = 0; t < n_tiles; ++t) {
        int r0, c0, h, w;
        tile_box(t, &r0, &c0, &h, &w);
        if (c0 > 0)
            for (int k = 0; k < h; ++k) edge.push_back({(r0 + k) * cols + c0, 0});
        if (r0 > 0)
            for (int k = 0; k < w; ++k) edge.push_back({r0 * cols + c0 + k, 1});
    }
    std::shuffle(edge.begin(), edge.end(), rng);
    for (const auto& e : edge) {
        if (L[(size_t)e.first] < 0) continue;
        const int r = e.first / cols, c = e.first % cols;
        if (e.second == 0) spx::det_border_left(L.data(), r, c, rows, cols);
        else spx::det_border_top(L.data(), r, c, rows, cols);
    }
    // flatten in a random order, then number the roots in raster order
    std::vector<int> cells;
    for (int i = 0; i < rows * cols; ++i)
        if (L[(size_t)i] >= 0) cells.push_back(i);
    std::shuffle(cells.begin(), cells.end(), rng);
    for (int i : cells) L[(size_t)i] = spx::det_find(L.data(), i);
    int n = 0;
    for (int i = 0; i < rows * cols; ++i)
        if (L[(size_t)i] == i) L[(size_t)i] = spx::det_encode_id(n++);
    for (int i = 0; i < rows * cols; ++i) labels_out[i] = spx::det_component(L.data(), i) + 1;
    return n;
}

// det_peak_key of each value at its index, so that the tests can check the key order against numpy's max / argmax
void emul_peak_keys(const float* v, const int* idx, int n, unsigned long long* out) {
    for (int i = 0; i < n; ++i) out[i] = spx::det_peak_key(v[i], idx[i]);
}

}
