// CPU harness of the multi-job DDC's work split (csrc/spx_ddc_device.cuh): the __host__ __device__ functions
// ddc_jobs_kernel uses to walk a CTA's run of sub-tiles job by job, run on the host so that tests/test_extract_cpu.py can
// check that every output of every job is computed exactly once.
#include "../../sdr_iq_visualizer_b200/csrc/spx_ddc_device.cuh"

extern "C" {

// CTA b of `grid` walks its run of the n = tile0[n_jobs] global sub-tiles job by job, as ddc_jobs_kernel does.  Writes
// one (cta, job, first local sub-tile, end local sub-tile) row per part to seg[cap][4] and returns the number of parts
// (at most cap are written).
long long emul_job_walk(const long long* tile0, int n_jobs, long long grid, long long* seg, long long cap) {
    long long n_seg = 0;
    for (long long b = 0; b < grid; ++b) {
        long long t, t1;
        spx::ddc_cta_run(b, grid, tile0[n_jobs], &t, &t1);
        while (t < t1) {
            int j;
            long long k0;
            const long long e = spx::ddc_segment(tile0, n_jobs, t, t1, &j, &k0);
            if (n_seg < cap) {
                long long* r = seg + 4 * n_seg;
                r[0] = b;
                r[1] = j;
                r[2] = k0;
                r[3] = k0 + (e - t);
            }
            ++n_seg;
            t = e;
        }
    }
    return n_seg;
}

}
