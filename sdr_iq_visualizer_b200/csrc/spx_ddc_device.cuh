// spx_ddc_device.cuh -- per-element math of the digital down-converter (K9, spx_ddc.cu), host and device.
//
// Kept apart from the kernel so that a CPU harness (tests/emul/ddc_emul.cu) runs exactly these functions.  Every product
// and sum is written out (fmaf, ddc_mul, ddc_add) so that no compiler contracts or reorders them: the host build and the
// device build give the same bits.
#pragma once
#include <math.h>
#include <stdint.h>

namespace spx {

__host__ __device__ inline float ddc_mul(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
__host__ __device__ inline float ddc_add(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}

// NCO phase of global sample n: n * phase_inc mod 2^64 (exact; depends on the global index only)
__host__ __device__ inline uint64_t ddc_phase(uint64_t n, uint64_t inc) { return n * inc; }

// (cos, sin) of 2 pi phi / 2^64.  The top 32 bits of the phase pick the nearest quadrant q and a residual angle a in
// [-pi/4, pi/4); sin a and cos a are their Taylor polynomials to a^9 / a^8 (truncation below 3e-8), and the quadrant is
// applied by swapping and negating.  Error against float64 is about 1e-7.
__host__ __device__ inline void ddc_cis(uint64_t phi, float* c_out, float* s_out) {
    const uint32_t u = (uint32_t)(phi >> 32);
    const uint32_t q = (u + 0x20000000u) >> 30;
    const int32_t rem = (int32_t)(u - (q << 30));
    const float a = ddc_mul((float)rem, 1.46291807926715968e-9f);   // 2 pi / 2^32
    const float a2 = ddc_mul(a, a);
    float s = fmaf(fmaf(fmaf(2.75573192e-6f, a2, -1.98412698e-4f), a2, 8.33333333e-3f), a2, -1.66666667e-1f);
    s = fmaf(ddc_mul(s, a2), a, a);
    float c = fmaf(fmaf(fmaf(fmaf(2.48015873e-5f, a2, -1.38888889e-3f), a2, 4.16666667e-2f), a2, -0.5f), a2, 1.0f);
    float co, si;
    switch (q) {
        case 0: co = c; si = s; break;
        case 1: co = -s; si = c; break;
        case 2: co = -c; si = -s; break;
        default: co = s; si = -c; break;
    }
    *c_out = co;
    *s_out = si;
}

// mixed sample: (xr + i xi) * exp(-2 pi i phi / 2^64)
__host__ __device__ inline void ddc_mix(float xr, float xi, uint64_t phi, float* re, float* im) {
    float c, s;
    ddc_cis(phi, &c, &s);
    *re = fmaf(xr, c, ddc_mul(xi, s));
    *im = fmaf(xi, c, -ddc_mul(xr, s));
}

// Work split of the FIR sum y[m] = sum_j g[j] mix[mD + j] (g = the taps reversed, g[j] = h[T - 1 - j]).
//   Lane l of a warp sums the taps j = l (mod 32); with c = D / gcd(D, 32) its taps are j = 32 (rho + c t) + l, and it
//   walks rho = wr, wr + WR, ... < c, t = 0, 1, ... in that order, one float32 fmaf chain per component.
//   The 32 lane sums are added as a tree: pairs (l, l + 16), then (l, l + 8), ... (l, l + 1).
//   The WR warps that share an output (wr = 0 .. WR - 1, each its own rho) are added in order of wr.
// Outputs m and m + s (s = 32 / gcd(D, 32)) read samples exactly lcm(D, 32) apart, so a lane slides one register
// window over the outputs m, m + s, m + 2s, ... .  Nothing here depends on where m falls in a tile or a call.
struct DdcGeom {
    int s;    // output stride of a lane's window
    int c;    // tap classes of one lane
    int wr;   // warps that split the classes of one output
    int wg;   // 8 / wr: warp groups of a CTA (8 warps)
};

__host__ __device__ inline DdcGeom ddc_geom(int D) {
    const int low = D & -D;
    const int g = low < 32 ? low : 32;
    DdcGeom G;
    G.s = 32 / g;
    G.c = D / g;
    int wr = 1;
    while (wr * 2 <= G.c && wr * 2 <= 8) wr *= 2;
    G.wr = wr;
    G.wg = 8 / wr;
    return G;
}

// taps t = 0 .. n - 1 of lane l in class rho: 32 (rho + c t) + l < T
__host__ __device__ inline int ddc_lane_taps(int T, int c, int lane, int rho) {
    const int j0 = 32 * rho + lane;
    return j0 >= T ? 0 : (T - 1 - j0) / (32 * c) + 1;
}

// Work split of a call.  The call's outputs are cut into sub-tiles of SUB outputs, and CTA b of `grid` takes the
// contiguous run [b n / grid, (b + 1) n / grid) of the n sub-tiles.
__host__ __device__ inline void ddc_cta_run(long long b, long long grid, long long n, long long* s0, long long* s1) {
    *s0 = b * n / grid;
    *s1 = (b + 1) * n / grid;
}

// Multi-job calls (spx_ddc_exec_jobs; the walk is run on the host by tests/emul/ddc_jobs_emul.cu): job j owns the global sub-tiles [tile0[j], tile0[j + 1]), ceil(n_out_j / SUB) of
// them, and tile0[n_jobs] is their total.  The job of global sub-tile t < tile0[n_jobs] is the largest j with
// tile0[j] <= t; a job without outputs owns no sub-tile and is never the answer.
__host__ __device__ inline int ddc_job_of(const long long* tile0, int n_jobs, long long t) {
    int lo = 0, hi = n_jobs;   // tile0[lo] <= t < tile0[hi]
    while (hi - lo > 1) {
        const int mid = lo + (hi - lo) / 2;
        if (tile0[mid] <= t) lo = mid;
        else hi = mid;
    }
    return lo;
}

// The part of a CTA's run [t, t1) that lies in one job: *job, its local first sub-tile *k0, and (returned) the global
// end of the part, where the CTA goes on with the next job.
__host__ __device__ inline long long ddc_segment(const long long* tile0, int n_jobs, long long t, long long t1, int* job,
                                                 long long* k0) {
    const int j = ddc_job_of(tile0, n_jobs, t);
    *job = j;
    *k0 = t - tile0[j];
    return tile0[j + 1] < t1 ? tile0[j + 1] : t1;
}

// tree sum of 32 lane partials (in place; the result is v[0])
__host__ __device__ inline float ddc_lane_tree(float* v) {
    for (int o = 16; o >= 1; o >>= 1)
        for (int l = 0; l < o; ++l) v[l] = ddc_add(v[l], v[l + o]);
    return v[0];
}

// Output m in the kernel's order, for the CPU harness.  mix_re / mix_im: the mixed samples mD .. mD + T - 1.
__host__ __device__ inline void ddc_output(const float* g, int T, int D, const float* mix_re, const float* mix_im, float* yr,
                                           float* yi) {
    const DdcGeom G = ddc_geom(D);
    float wre = 0.f, wim = 0.f;
    for (int w = 0; w < G.wr; ++w) {
        float pr[32], pi[32];
        for (int l = 0; l < 32; ++l) {
            float ar = 0.f, ai = 0.f;
            for (int rho = w; rho < G.c; rho += G.wr) {
                const int n = ddc_lane_taps(T, G.c, l, rho);
                for (int t = 0; t < n; ++t) {
                    const int j = 32 * (rho + G.c * t) + l;
                    ar = fmaf(g[j], mix_re[j], ar);
                    ai = fmaf(g[j], mix_im[j], ai);
                }
            }
            pr[l] = ar;
            pi[l] = ai;
        }
        const float r = ddc_lane_tree(pr), i = ddc_lane_tree(pi);
        wre = w == 0 ? r : ddc_add(wre, r);
        wim = w == 0 ? i : ddc_add(wim, i);
    }
    *yr = wre;
    *yi = wim;
}

}  // namespace spx
