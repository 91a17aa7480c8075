// CPU harness of the DDC math (csrc/spx_ddc_device.cuh): the __host__ __device__ functions K9 uses, run on the host so
// that tests/test_ddc_cpu.py can hold them to tests/ddc_ref.py and the GPU tests can compare K9 with them bit for bit.
#include <vector>

#include "../../sdr_iq_visualizer_b200/csrc/spx_ddc_device.cuh"

extern "C" {

void emul_cis(const unsigned long long* phi, long long n, float* c, float* s) {
    for (long long i = 0; i < n; ++i) spx::ddc_cis(phi[i], &c[i], &s[i]);
}

// the full definition in the kernel's order: x interleaved float32 (fmt 0) or int16 (fmt 1), taps h[0 .. T - 1] float32
void emul_ddc(const void* x, int fmt, float scale, long long L, unsigned long long first_sample, unsigned long long inc,
              const float* h, int T, int D, float* out) {
    if (L < T) return;
    std::vector<float> mr((size_t)L), mi((size_t)L), g((size_t)T);
    for (long long n = 0; n < L; ++n) {
        const float xr = fmt ? (float)((const short*)x)[2 * n] : ((const float*)x)[2 * n];
        const float xi = fmt ? (float)((const short*)x)[2 * n + 1] : ((const float*)x)[2 * n + 1];
        spx::ddc_mix(spx::ddc_mul(xr, scale), spx::ddc_mul(xi, scale), spx::ddc_phase(first_sample + (unsigned long long)n, inc),
                     &mr[(size_t)n], &mi[(size_t)n]);
    }
    for (int j = 0; j < T; ++j) g[(size_t)j] = h[T - 1 - j];
    const long long M = (L - T) / D + 1;
    for (long long m = 0; m < M; ++m)
        spx::ddc_output(g.data(), T, D, mr.data() + m * D, mi.data() + m * D, &out[2 * m], &out[2 * m + 1]);
}

void emul_geom(int D, int* out4) {
    const spx::DdcGeom G = spx::ddc_geom(D);
    out4[0] = G.s;
    out4[1] = G.c;
    out4[2] = G.wr;
    out4[3] = G.wg;
}

}
