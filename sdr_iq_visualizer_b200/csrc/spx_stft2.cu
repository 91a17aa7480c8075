// N = 1024 / 2048 / 4096 instantiations of K1v2 (warp-local first exchange, one block barrier per frame, swizzled TMA
// tensor staging).  See spx_stft2_kernel.cuh / spx_stft2_device.cuh.
#include "spx_stft2_kernel.cuh"

namespace spx {

tmap_encode_fn tmap_encoder() {
    static tmap_encode_fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (tmap_encode_fn)p;
        else
            cudaGetLastError();
        tried = true;
    }
    return fn;
}

// Default kernels with the set of row outputs fixed at compile time (uint8 rows only / f32 dB rows only / accumulators only /
// read from the parameters): as run-time branches in the frame loop the unused outputs cost registers and 1 - 2 % (measured on
// config 2: 106.2 -> 107.8 GS/s).
template <int N, int FMT, int TUNE>
static int launch_acc(StftLaunch& L, bool acc) {
    return acc ? launch_stft2_inst<N, FMT, true, 2, TUNE>(L) : launch_stft2_inst<N, FMT, false, 2, TUNE>(L);
}
template <int N, int FMT, int TUNE>
static int launch_outs(StftLaunch& L) {
    const bool acc = L.p.welch_acc != nullptr || L.p.maxhold != nullptr;
    const bool wf = L.p.wf_rows != nullptr, db = L.p.db_rows != nullptr, spec = L.p.spec_rows != nullptr;
    if (wf && !db && !spec) return launch_acc<N, FMT, TUNE | TUNE_ONLY_U8>(L, acc);
    if (db && !wf && !spec) return launch_acc<N, FMT, TUNE | TUNE_ONLY_DB>(L, acc);
    if (acc && !wf && !db && !spec) return launch_stft2_inst<N, FMT, true, 2, TUNE | TUNE_NO_ROWS>(L);
    return launch_acc<N, FMT, TUNE>(L, acc);
}
template <int N, int TUNE>
static int launch_fmt_outs(StftLaunch& L) {
    return L.in_fmt == FMT_CF32 ? launch_outs<N, FMT_CF32, TUNE>(L) : launch_outs<N, FMT_CI16, TUNE>(L);
}

int launch_stft2(StftLaunch& L) {
    // FMA-form DFTs + uint8 index on the FMA / ALU pipes instead of F2I (XU)
    constexpr int T0 = TUNE_I2FP | TUNE_FMADFT | TUNE_QFMA;
    if (L.variant == 22) {   // the generic T0 kernel alone: the reference the strip kernel is tested against
        switch (L.nfft) {
            case 1024: return launch_stft2_n<1024, 2, T0>(L);
            case 2048: return launch_stft2_n<2048, 2, T0>(L);
            case 4096: return launch_stft2_n<4096, 2, T0>(L);
        }
    }
    if (L.nfft == 4096 && L.in_fmt == FMT_CF32 && L.p.hop == 1024) {
        // measured (profiles/r02_strip_staging_sweep.jsonl): strip staging wins 3 % on cf32 at 75 % overlap (the frame is
        // 32 KB, three quarters of it already in shared memory), is neutral for ci16 and at 50 % overlap -- used only here
        return launch_stft2_strip<T0>(L);
    }
    // L2 prefetch of the next frame (compile-time as well): cf32, N = 4096 without overlap only (+ 5 %,
    // profiles/r02_l2_prefetch_sweep.txt; neutral for int16, - 1 % with overlap, - 3 % for N = 2048 / 1024 with their 2 / 4
    // frames in flight per CTA)
    if (L.nfft == 4096 && L.in_fmt == FMT_CF32 && L.p.hop >= 4096) return launch_outs<4096, FMT_CF32, T0 | TUNE_L2PF>(L);
    switch (L.nfft) {
        case 1024: return launch_fmt_outs<1024, T0>(L);
        case 2048: return launch_fmt_outs<2048, T0>(L);
        case 4096: return launch_fmt_outs<4096, T0>(L);
        default: return spx_set_error(SPX_E_UNSUPPORTED, "K1v2 handles nfft 1024 / 2048 / 4096, not %d", L.nfft);
    }
}

}  // namespace spx
