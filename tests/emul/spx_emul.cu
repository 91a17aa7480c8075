// spx_emul.cu -- TEST INFRASTRUCTURE ONLY.  Re-executes the per-thread phases of the CUDA STFT kernel
// (sdr_iq_visualizer_b200/csrc/spx_stft_device.cuh, the exact code the GPU runs) on the CPU, thread
// by thread and barrier by barrier, so that the `-m "not gpu"` tests can check the Stockham index
// maps, padding, twiddle tables and epilogue against the numpy oracle without a GPU.
// It is never linked into libspx and never imported by the product package.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "../../sdr_iq_visualizer_b200/csrc/spx_stft_device.cuh"
#include "../../sdr_iq_visualizer_b200/csrc/spx_stft2_device.cuh"
#include "../../sdr_iq_visualizer_b200/csrc/spx_big2_device.cuh"
#include "../../sdr_iq_visualizer_b200/csrc/spx_tables.h"

using namespace spx;

static bool g_staged = false;  // emulate the bulk-copy staging buffer (pass 0 reads shared memory)

template <int N, int FMT, bool ACC, int TWM, int S>
static void run_phase(std::vector<float2>& v, StftParams& p, long long s0, long long row, float2* A, float2* B,
                      const float2* tw, std::vector<TwRegs<N>>& twr, std::vector<StftAcc<ACC>>& acc) {
    constexpr int T = N / 16;
    std::vector<unsigned char> stage;
    const void* st = nullptr;
    if (S == 0 && g_staged) {
        const size_t elt = FMT == FMT_CF32 ? 8 : 4;
        stage.resize((size_t)N * elt);
        memcpy(stage.data(), (const char*)p.in + (size_t)s0 * elt, stage.size());
        st = stage.data();
    }
    for (int tid = 0; tid < T; ++tid)
        stft_phase<N, FMT, ACC, TWM, S>(&v[(size_t)tid * 16], tid, p, s0, row, true, A, B, tw, twr[tid], acc[tid], st,
                                        st ? p.win : nullptr);  // first N/2 entries of the global table = the half table
}

template <int N, int FMT, bool ACC, int TWM>
static int emul_stft(StftParams p) {
    constexpr int T = N / 16, P = plan_passes(N);
    std::vector<float2> tw = build_twiddles(N);
    p.tw = tw.data();
    std::vector<float2> A((size_t)padded_size(N)), B((size_t)N), v((size_t)T * 16);
    std::vector<TwRegs<N>> twr((size_t)T);
    std::vector<StftAcc<ACC>> acc((size_t)T);
    if constexpr (TWM == TW_REG && P > 1) {
        for (int tid = 0; tid < T; ++tid) {
            if constexpr (P > 1) tw_regs_load_pass<N, 1>(twr[tid], tid, p.tw);
            if constexpr (P > 2) tw_regs_load_pass<N, 2>(twr[tid], tid, p.tw);
            if constexpr (P > 3) tw_regs_load_pass<N, 3>(twr[tid], tid, p.tw);
        }
    }
    for (auto& a : acc) a.reset();
    const long long F = p.frames_per_stream;
    for (long long chunk = 0; chunk < p.total_chunks; ++chunk) {
        const long long stream = chunk / p.chunks_per_stream;
        const long long f0 = (chunk - stream * p.chunks_per_stream) * p.frames_per_chunk;
        long long nf = F - f0;
        if (nf > p.frames_per_chunk) nf = p.frames_per_chunk;
        for (long long fi = 0; fi < nf; ++fi) {
            const long long s0 = stream * p.stream_stride + (f0 + fi) * p.hop;
            const long long row = stream * F + f0 + fi;
            run_phase<N, FMT, ACC, TWM, 0>(v, p, s0, row, A.data(), B.data(), p.tw, twr, acc);
            if constexpr (P > 1) run_phase<N, FMT, ACC, TWM, 1>(v, p, s0, row, A.data(), B.data(), p.tw, twr, acc);
            if constexpr (P > 2) run_phase<N, FMT, ACC, TWM, 2>(v, p, s0, row, A.data(), B.data(), p.tw, twr, acc);
            if constexpr (P > 3) run_phase<N, FMT, ACC, TWM, 3>(v, p, s0, row, A.data(), B.data(), p.tw, twr, acc);
        }
        if constexpr (ACC) {
            for (int tid = 0; tid < T; ++tid) {
                for (int i = 0; i < 16; ++i) {
                    const long long o = stream * N + acc_pos<N>(tid, i);
                    if (p.welch_acc) p.welch_acc[o] += (double)acc[tid].sum[i];
                    if (p.maxhold && acc[tid].mx[i] > p.maxhold[o]) p.maxhold[o] = acc[tid].mx[i];
                }
                acc[tid].reset();
            }
        }
    }
    return 0;
}

template <int N, int TWM>
static int emul_n(int fmt, bool acc, StftParams& p) {
    if (fmt == FMT_CF32) return acc ? emul_stft<N, FMT_CF32, true, TWM>(p) : emul_stft<N, FMT_CF32, false, TWM>(p);
    return acc ? emul_stft<N, FMT_CI16, true, TWM>(p) : emul_stft<N, FMT_CI16, false, TWM>(p);
}

// ------------------------------------------------------------------ K1v2 (warp-local first exchange), same contract
template <int N, int FMT, bool ACC, int TUNE>
static int emul_stft2(StftParams p) {
    using G = Stft2Geom<N>;
    constexpr int T = G::T;
    constexpr bool TWC_REGS = G::C == 16;
    constexpr size_t ELT = FMT == FMT_CF32 ? 8 : 4;
    std::vector<float2> tw = build_twiddles(N);
    p.tw = tw.data();
    std::vector<float2> X[2] = {std::vector<float2>((size_t)G::X_F2), std::vector<float2>((size_t)G::X_F2)};
    std::vector<float2> v((size_t)T * 16);
    std::vector<TwRegs<N>> twr((size_t)T);
    std::vector<StftAcc<ACC>> acc((size_t)T);
    std::vector<float> wtab((size_t)N / 2);
    std::vector<unsigned char> stage((size_t)N * ELT);
    for (int tid = 0; tid < T; ++tid) {
        // phase B uses the pass-1 bases of k_a = lane & 15, phase C the pass-2 bases of j = tid: a thread needs both
        TwRegs<N> b1;
        tw_regs_load_pass<N, 1>(b1, k2_ka_of(tid), p.tw);
        if constexpr (TWC_REGS) tw_regs_load_pass<N, 2>(b1, tid, p.tw);
        twr[tid] = b1;
        if (p.win) k2_build_window<N>(wtab.data(), p.win, tid);
    }
    for (auto& a : acc) a.reset();
    const long long F = p.frames_per_stream;
    int par = 0;
    for (long long chunk = 0; chunk < p.total_chunks; ++chunk) {
        const long long stream = chunk / p.chunks_per_stream;
        const long long f0 = (chunk - stream * p.chunks_per_stream) * p.frames_per_chunk;
        long long nf = F - f0;
        if (nf > p.frames_per_chunk) nf = p.frames_per_chunk;
        for (long long fi = 0; fi < nf; ++fi) {
            const long long s0 = stream * p.stream_stride + (f0 + fi) * p.hop;
            const long long row = stream * F + f0 + fi;
            // what the TMA tensor copy with CU_TENSOR_MAP_SWIZZLE_128B leaves in shared memory
            const unsigned char* src = (const unsigned char*)p.in + (size_t)s0 * ELT;
            for (unsigned byte = 0; byte < N * ELT; byte += 16) memcpy(&stage[swz128(byte)], src + byte, 16);
            float2* Xp = X[par].data();
            for (int tid = 0; tid < T; ++tid) k2_phase_a<N, FMT, TUNE>(&v[(size_t)tid * 16], tid, stage.data(), p.win ? wtab.data() : nullptr, Xp);
            for (int tid = 0; tid < T; ++tid) k2_phase_b1<N, TUNE>(&v[(size_t)tid * 16], tid, Xp, twr[tid]);
            for (int tid = 0; tid < T; ++tid) k2_phase_b2<N>(&v[(size_t)tid * 16], tid, Xp);
            for (int tid = 0; tid < T; ++tid)
                k2_phase_c<N, ACC, TWC_REGS, TUNE>(&v[(size_t)tid * 16], tid, Xp, p, row, p.tw, twr[tid], acc[tid]);
            par ^= 1;
        }
        if constexpr (ACC) {
            for (int tid = 0; tid < T; ++tid) {
                for (int i = 0; i < 16; ++i) {
                    const long long o = stream * N + acc_pos<N>(tid, i);
                    if (p.welch_acc) p.welch_acc[o] += (double)acc[tid].sum[i];
                    if (p.maxhold && acc[tid].mx[i] > p.maxhold[o]) p.maxhold[o] = acc[tid].mx[i];
                }
                acc[tid].reset();
            }
        }
    }
    return 0;
}

template <int N, int TUNE>
static int emul2_n(int fmt, bool acc, StftParams& p) {
    if (fmt == FMT_CF32) return acc ? emul_stft2<N, FMT_CF32, true, TUNE>(p) : emul_stft2<N, FMT_CF32, false, TUNE>(p);
    return acc ? emul_stft2<N, FMT_CI16, true, TUNE>(p) : emul_stft2<N, FMT_CI16, false, TUNE>(p);
}
template <int TUNE>
static int emul2_nfft(int nfft, int fmt, bool acc, StftParams& p) {
    switch (nfft) {
        case 1024: return emul2_n<1024, TUNE>(fmt, acc, p);
        case 2048: return emul2_n<2048, TUNE>(fmt, acc, p);
        case 4096: return emul2_n<4096, TUNE>(fmt, acc, p);
        default: return -4;
    }
}

extern "C" int spx_emul_stft(int nfft, int in_fmt, int tw_mode, const void* in, long long n_samples, int n_streams,
                             long long stream_stride, int hop, const float* win, float db_eps, float vmin, float vmax,
                             int frames_per_chunk, float* db_rows, unsigned char* wf_rows, float* spec_rows,
                             double* welch_acc, float* maxhold) {
    StftParams p;
    memset(&p, 0, sizeof(p));
    p.in = in;
    p.stream_stride = stream_stride;
    p.n_streams = n_streams;
    p.hop = hop;
    p.frames_per_stream = n_samples < nfft ? 0 : (n_samples - nfft) / hop + 1;
    p.win = win;
    p.db_rows = db_rows;
    p.wf_rows = wf_rows;
    p.spec_rows = reinterpret_cast<float2*>(spec_rows);
    p.welch_acc = welch_acc;
    p.maxhold = maxhold;
    p.db_eps = db_eps;
    p.db_pw_min = db_eps * db_eps * 1099511627776.0f;  // (2^20 eps)^2
    p.q_a = (float)(3.01029995663981195214 * 256.0 / ((double)vmax - (double)vmin));  // 10 log10(2) * scale
    p.q_b = (float)(-(double)vmin * 256.0 / ((double)vmax - (double)vmin));
    if (p.frames_per_stream == 0) return 0;
    p.frames_per_chunk = frames_per_chunk;
    p.chunks_per_stream = (int)((p.frames_per_stream + frames_per_chunk - 1) / frames_per_chunk);
    p.total_chunks = (long long)p.chunks_per_stream * n_streams;
    const bool acc = welch_acc != nullptr || maxhold != nullptr;
    if (tw_mode & 0x20) {   // K1v2 phases; 0x40: FMA-form DFTs + FMA-pipe colormap index, 0x80: FMA-form DFTs + F2I index
        if (tw_mode & 0x40) return emul2_nfft<TUNE_FMADFT | TUNE_QFMA>(nfft, in_fmt, acc, p);
        if (tw_mode & 0x80) return emul2_nfft<TUNE_FMADFT>(nfft, in_fmt, acc, p);
        return emul2_nfft<0>(nfft, in_fmt, acc, p);
    }
    g_staged = (tw_mode & 0x10) != 0;
    tw_mode &= 0xf;
#define CASE(NN)                                                                  \
    case NN:                                                                      \
        if (tw_mode == TW_REG) {                                                  \
            if constexpr (NN == 256 || NN == 4096) return emul_n<NN, TW_REG>(in_fmt, acc, p); \
            return -4;                                                            \
        }                                                                         \
        return emul_n<NN, TW_LDG>(in_fmt, acc, p);
    switch (nfft) {
        CASE(16) CASE(32) CASE(64) CASE(128) CASE(256) CASE(512) CASE(1024) CASE(2048) CASE(4096) CASE(8192)
        default: return -4;
    }
#undef CASE
}

// ------------------------------------------------------------------ K2v2: single-kernel 65536-point STFT, role by role
template <bool ACC, int TUNE, int FMT = FMT_CF32>
static int emul_big2(const void* in_any, long long n_samples, int hop, const float* win, float db_eps, float vmin, float vmax,
                     unsigned char* wf_rows, double* welch_acc, float* maxhold) {
    const float2* in = reinterpret_cast<const float2*>(in_any);
    const unsigned int* in16 = reinterpret_cast<const unsigned int*>(in_any);   // one ci16 sample = 4 bytes
    constexpr int N = BIG2_N;
    using G = Stft2Geom<4096>;
    const long long F = n_samples < N ? 0 : (n_samples - N) / hop + 1;
    std::vector<float2> tw = build_twiddles(4096);      // pass-1 bases W_256^{b k_a} live in the N = 4096 table
    std::vector<float2> bases((size_t)16 * 7 * 256);
    const double two_pi = 6.283185307179586476925286766559;
    for (int g = 0; g < 16; ++g)
        for (int tid = 0; tid < 256; ++tid) {
            unsigned e[7];
            big2_base_exponents(g, tid, e);
            for (int q = 0; q < 7; ++q) {
                const double a = -two_pi * (double)e[q] / (double)N;
                bases[((size_t)g * 7 + q) * 256 + tid] = make_float2((float)cos(a), (float)sin(a));
            }
        }
    std::vector<TwRegs<4096>> twr(256);
    for (int tid = 0; tid < 256; ++tid) tw_regs_load_pass<4096, 1>(twr[tid], k2_ka_of(tid), tw.data());
    std::vector<float2> T((size_t)N), X((size_t)G::X_F2), v((size_t)256 * 16);
    std::vector<unsigned char> stage((size_t)256 * 128), u8tile((size_t)256 * 16);
    std::vector<float> wfull((size_t)16 * 256);
    std::vector<std::vector<StftAcc<ACC>>> acc(16, std::vector<StftAcc<ACC>>(256));
    for (auto& a : acc) for (auto& t : a) t.reset();
    const float q_a = (float)(3.01029995663981195214 * 256.0 / ((double)vmax - (double)vmin));
    const float q_b = (float)(-(double)vmin * 256.0 / ((double)vmax - (double)vmin));
    const float pw_min = db_eps * db_eps * 1099511627776.0f;
    for (long long f = 0; f < F; ++f) {
        const float2* x = in + f * hop;
        const unsigned int* x16 = in16 + f * hop;
        for (int g = 0; g < 16; ++g) {   // role A of every column tile
            for (int n1 = 0; n1 < 256; ++n1) {    // what the swizzled TMA box leaves in shared memory: {128 B, 256 rows} / ci16: {64 B, 256 rows}
                if (FMT == FMT_CF32)
                    for (int ch = 0; ch < 8; ++ch) memcpy(&stage[swz128((unsigned)(128 * n1 + 16 * ch))], x + 256 * n1 + 16 * g + 2 * ch, 16);
                else
                    for (int ch = 0; ch < 4; ++ch) memcpy(&stage[swz64((unsigned)(64 * n1 + 16 * ch))], x16 + 256 * n1 + 16 * g + 4 * ch, 16);
            }
            for (int tid = 0; tid < 256; ++tid) {
                float w[16];
                if (win) for (int a = 0; a < 16; ++a) w[a] = win[big2_sample_of(g, a, tid)];
                if (FMT == FMT_CF32) {
                    big2_phase_a<TUNE, 1>(&v[(size_t)tid * 16], tid, stage.data(), win ? w : nullptr, X.data());
                } else {
                    big2_load_tile_ci16<1>(&v[(size_t)tid * 16], tid, stage.data(), win ? w : nullptr);
                    big2_dft_store(&v[(size_t)tid * 16], tid, X.data());
                }
            }
            for (int tid = 0; tid < 256; ++tid) k2_phase_b1<4096, TUNE>(&v[(size_t)tid * 16], tid, X.data(), twr[tid]);
            for (int tid = 0; tid < 256; ++tid)
                big2_twiddle_store<TUNE>(&v[(size_t)tid * 16], tid, &bases[(size_t)g * 7 * 256], T.data() + (size_t)g * 16 * 256);
        }
        for (int g = 0; g < 16; ++g) {   // role B of every row tile
            for (int n2 = 0; n2 < 256; ++n2)
                for (int ch = 0; ch < 8; ++ch) memcpy(&stage[swz128((unsigned)(128 * n2 + 16 * ch))], &T[(size_t)n2 * 256 + 16 * g + 2 * ch], 16);
            for (int tid = 0; tid < 256; ++tid) big2_phase_a<TUNE>(&v[(size_t)tid * 16], tid, stage.data(), nullptr, X.data());
            for (int tid = 0; tid < 256; ++tid) k2_phase_b1<4096, TUNE>(&v[(size_t)tid * 16], tid, X.data(), twr[tid]);
            for (int tid = 0; tid < 256; ++tid)
                big2_epilogue<ACC, TUNE>(&v[(size_t)tid * 16], tid, db_eps, pw_min, q_a, q_b, wf_rows != nullptr, acc[g][tid], u8tile.data());
            if (wf_rows)
                for (int k2s = 0; k2s < 256; ++k2s) memcpy(wf_rows + (size_t)f * N + 256 * k2s + 16 * g, &u8tile[(size_t)16 * k2s], 16);
        }
    }
    if constexpr (ACC) {
        for (int g = 0; g < 16; ++g)
            for (int tid = 0; tid < 256; ++tid)
                for (int kb = 0; kb < 16; ++kb) {
                    const int o = big2_acc_pos(g, tid, kb);
                    if (welch_acc) welch_acc[o] += (double)acc[g][tid].sum[kb];
                    if (maxhold && acc[g][tid].mx[kb] > maxhold[o]) maxhold[o] = acc[g][tid].mx[kb];
                }
    }
    return 0;
}

extern "C" int spx_emul_big2(const void* in, long long n_samples, int hop, const float* win, float db_eps, float vmin, float vmax,
                             int tune, unsigned char* wf_rows, double* welch_acc, float* maxhold) {
    const bool acc = welch_acc != nullptr || maxhold != nullptr;
    const void* x = in;
    if (tune) return acc ? emul_big2<true, TUNE_FMADFT | TUNE_QFMA>(x, n_samples, hop, win, db_eps, vmin, vmax, wf_rows, welch_acc, maxhold)
                         : emul_big2<false, TUNE_FMADFT | TUNE_QFMA>(x, n_samples, hop, win, db_eps, vmin, vmax, wf_rows, welch_acc, maxhold);
    return acc ? emul_big2<true, TUNE_FMADFT>(x, n_samples, hop, win, db_eps, vmin, vmax, wf_rows, welch_acc, maxhold)
               : emul_big2<false, TUNE_FMADFT>(x, n_samples, hop, win, db_eps, vmin, vmax, wf_rows, welch_acc, maxhold);
}

extern "C" int spx_emul_big2_ci16(const void* in, long long n_samples, int hop, const float* win, float db_eps, float vmin, float vmax,
                                  unsigned char* wf_rows, double* welch_acc, float* maxhold) {
    const bool acc = welch_acc != nullptr || maxhold != nullptr;
    return acc ? emul_big2<true, TUNE_FMADFT | TUNE_QFMA, FMT_CI16>(in, n_samples, hop, win, db_eps, vmin, vmax, wf_rows, welch_acc, maxhold)
               : emul_big2<false, TUNE_FMADFT | TUNE_QFMA, FMT_CI16>(in, n_samples, hop, win, db_eps, vmin, vmax, wf_rows, welch_acc, maxhold);
}

// plan introspection for the tests
extern "C" int spx_emul_plan(int nfft, int* radices /*[5]*/, int* tw_size) {
    const int p = plan_passes(nfft);
    for (int s = 0; s < 5; ++s) radices[s] = plan_radix(nfft, s);
    *tw_size = plan_tw_size(nfft);
    return p;
}
