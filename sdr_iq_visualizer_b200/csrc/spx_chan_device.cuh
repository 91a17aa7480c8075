// spx_chan_device.cuh -- per-thread fold and index maps of the polyphase channelizer (K10, spx_chan.cu), host and device.
//
// Channel j (fftshift order, c = j - M/2) of output m is
//   y_j[m] = sum_r v_m[r] exp(-2 pi i c r / M),   v_m[r] = sum_{k : (first_sample + mD + T-1-k) mod M = r} h[k] x[mD + T-1-k]
// i.e. an M-point forward DFT of the fold v_m read out in fftshift order (the STFT epilogue's shift_off / out_bin maps).
// With g[j] = h[T - 1 - j] (the taps reversed) and window offset j = n - mD, sample n belongs to class
// r = (first_sample + mD + j) mod M, so class r holds the offsets j = j_r, j_r + M, j_r + 2M, ... < T with
// j_r = (r - cls0) mod M, cls0 = (first_sample + mD) mod M.  The fold sums them in that order (ascending j), one float32
// fmaf chain per component; the DFT is the STFT's per-pass Stockham code (spx_stft_device.cuh).  Nothing depends on where
// m falls in a tile or a call.
//
// Kept apart from the kernel so that a CPU harness (tests/emul/chan_emul.cu) runs exactly these functions.
#pragma once
#include "spx_ddc_device.cuh"
#include "spx_stft_device.cuh"

namespace spx {

// global class of the first sample of output m's window: (first_sample + m D) mod M
SPX_HD unsigned chan_cls0(unsigned long long n0, long long m, int D, int M) {
    return (unsigned)((n0 + (unsigned long long)m * (unsigned long long)D) & (unsigned long long)(M - 1));
}

// Fold of one FFT thread over the window offsets [j_lo, j_hi): v[t] += the terms of class r = ft + t M/16 (the FFT's
// pass-0 input layout, load_frame's index map) in that range, in ascending j, each component one fmaf chain continued from
// v[t].  Folding [0, T) at once, or [0, a), [a, b), ... [z, T) in turn from v = 0, gives the same bits.
// `x` holds samples in a ring of ring_n slots; window offset j sits in slot base + j, minus ring_n if that is >= ring_n
// (base + j_lo >= 0, base + j < 2 ring_n and j_hi - j_lo <= ring_n).
template <int M>
SPX_HD void chan_fold(float2* v, int ft, const float* g, int j_lo, int j_hi, const float2* x, int ring_n, int base,
                      unsigned cls0) {
    constexpr int TPF = M / 16;
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        const int r = ft + t * TPF;
        int j = (int)(((unsigned)r - cls0) & (unsigned)(M - 1));   // first offset of class r
        if (j < j_lo) j += (j_lo - j + M - 1) / M * M;
        float ar = v[t].x, ai = v[t].y;
        if (j < j_hi) {
            int s = base + j;
            if (s >= ring_n) s -= ring_n;
            for (; j < j_hi; j += M) {
                const float2 xv = x[s];
                const float gv = g[j];
                ar = fmaf(gv, xv.x, ar);
                ai = fmaf(gv, xv.y, ai);
                s += M;
                if (s >= ring_n) s -= ring_n;
            }
        }
        v[t] = make_float2(ar, ai);
    }
}

// channel (fftshift order) held in v[u R + t] of FFT thread ft after the last pass
template <int M>
SPX_HD int chan_of(int ft, int u, int t) {
    return shift_off<M>(t) + ft + (M / 16) * u;
}

// Pass S >= 1 of the M-point FFT of one frame for FFT thread ft: read pass S - 1's result from the exchange buffer `buf`
// (padded_size(M) float2), twiddle, DFT.  The kernel brackets it with block barriers; the host harness runs each pass over
// all threads in turn (chan_fft_host).
template <int M, int S>
SPX_HD void chan_pass(float2* v, int ft, float2* buf, const float2* tw) {
    pass_load_smem<M, S>(v, ft, buf);
    pass_twiddle_table<M, S, false>(v, ft, tw);
    pass_dft<M, S>(v);
}

// The whole M-point DFT of a fold on the host, phase by phase over the M/16 threads, with the kernel's pass code:
// fold[r] natural order in, out[j] fftshift order out.
template <int M>
__host__ inline void chan_fft_host(const float2* fold, const float2* tw, float2* out) {
    constexpr int TPF = M / 16, P = plan_passes(M);
    static_assert(P <= 4, "M <= 4096");
    float2 v[TPF][16];
    float2 buf[padded_size(M)];
    for (int ft = 0; ft < TPF; ++ft) {
        for (int t = 0; t < 16; ++t) v[ft][t] = fold[ft + t * TPF];
        pass_dft<M, 0>(v[ft]);
    }
    if constexpr (P > 1) {
        for (int ft = 0; ft < TPF; ++ft) pass_store_smem<M, 0>(v[ft], ft, buf);
        for (int ft = 0; ft < TPF; ++ft) chan_pass<M, 1>(v[ft], ft, buf, tw);
    }
    if constexpr (P > 2) {
        for (int ft = 0; ft < TPF; ++ft) pass_store_smem<M, 1>(v[ft], ft, buf);
        for (int ft = 0; ft < TPF; ++ft) chan_pass<M, 2>(v[ft], ft, buf, tw);
    }
    if constexpr (P > 3) {
        for (int ft = 0; ft < TPF; ++ft) pass_store_smem<M, 2>(v[ft], ft, buf);
        for (int ft = 0; ft < TPF; ++ft) chan_pass<M, 3>(v[ft], ft, buf, tw);
    }
    constexpr int R = plan_radix(M, P - 1), NB = 16 / R;
    for (int ft = 0; ft < TPF; ++ft)
        for (int u = 0; u < NB; ++u)
            for (int t = 0; t < R; ++t) out[chan_of<M>(ft, u, t)] = v[ft][u * R + t];
}

}  // namespace spx
