// CPU harness of the pooled-spectrogram math (csrc/spx_pool_device.cuh): the __host__ __device__ functions the kernels
// use, run on the host over arrays so that tests/test_pooled_cpu.py can hold them to tests/pool_ref.py.
#include "../../sdr_iq_visualizer_b200/csrc/spx_pool_device.cuh"

extern "C" {

void emul_db_to_power(const float* d, long long n, float eps, float* out) {
    for (long long i = 0; i < n; ++i) out[i] = spx::pool_db_to_power(d[i], eps);
}

void emul_mean_db(const double* sum, const long long* n_frames, long long n, int bins_per_col, float eps, float* out) {
    for (long long i = 0; i < n; ++i) out[i] = spx::pool_mean_db(sum[i], n_frames[i], bins_per_col, eps);
}

void emul_max_db(const double* acc, long long n, float* out) {
    for (long long i = 0; i < n; ++i) out[i] = spx::pool_max_db(acc[i]);
}

void emul_level(const float* db, long long n, float vmin, float vmax, unsigned char* out) {
    for (long long i = 0; i < n; ++i) out[i] = spx::pool_level(db[i], vmin, vmax);
}

long long emul_row_of(long long frame, long long k) { return spx::pool_row_of(frame, k); }
int emul_col_of(int bin, int b) { return spx::pool_col_of(bin, b); }
long long emul_row_frames(long long g, long long k, long long f_total) { return spx::pool_row_frames(g, k, f_total); }

}
