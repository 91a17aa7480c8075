// spx_stft_device.cuh -- per-thread phases of the fused STFT kernel (K1).
//
// One frame = unpack (int16|cf32) -> window -> Stockham FFT -> |X|^2 -> dB -> fftshift ->
// {f32 dB row, u8 waterfall row, Welch sum, max-hold}.  Replaces, fused and batched, the three
// lines /root/reference/app/sdr/streamer.py:119-121 and the mlab.psd frame loop behind
// /root/reference/scripts/process_sigmf_data.py:188 (SURVEY.md section 8(a) rows A1-A8).
//
// Everything here is __host__ __device__: the CUDA kernel (spx_stft.cu) and the CPU
// re-execution used by the `-m "not gpu"` tests (csrc/emul) share this code verbatim.
#pragma once
#include "spx_fft_core.cuh"

namespace spx {

enum { FMT_CF32 = 0, FMT_CI16 = 1 };
enum { TW_LDG = 0, TW_REG = 1, TW_SMEM = 2 };

struct StftParams {
    const void* in;              // cf32 (float2) or ci16 (short2) samples
    long long stream_stride;     // samples between consecutive streams
    long long frames_per_stream; // F
    int n_streams;
    int hop;
    const float* win;            // [N] window * in_scale, or nullptr (rect, scale 1)
    const float2* tw;            // twiddle table, plan_tw_size(N) entries
    float* db_rows;              // [n_streams*F][N] dB rows (fftshift order) or nullptr
    unsigned char* wf_rows;      // [n_streams*F][N] u8 colormap indices or nullptr
    float2* spec_rows;           // [n_streams*F][N] complex spectrum (fftshift order) or nullptr
    double* welch_acc;           // [n_streams][N]  += sum_f |X|^2   (fftshift order) or nullptr
    float* maxhold;              // [n_streams][N]  max= |X|^2       (fftshift order) or nullptr
    float db_eps;                // 20*log10(|X| + db_eps)
    float db_pw_min;             // below this |X|^2 the eps term matters and the exact form is evaluated
    float q_a, q_b;              // u8 = sat(floor((dB - vmin) * 256/(vmax-vmin))) evaluated on y = log2|X|^2: q_a * y + q_b
    int sys_atomics;             // accumulators may live on a peer GPU: flush with system-scope atomics
    int frames_per_chunk;        // accumulator flush granularity (<= 256)
    int chunks_per_stream;
    long long total_chunks;
};

// ------------------------------------------------------------------ device/host primitives
SPX_HD float2 ld_stream_cf32(const float2* p) {
#ifdef __CUDA_ARCH__
    float2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
    return r;
#else
    return *p;
#endif
}
// kernel tuning bits (template parameter TUNE).  FMADFT: radix-16 DFTs in FMA form (dft16_fma).  QFMA: the uint8 colormap
// index is produced on the FMA / ALU pipes (saturating FMA, min, round-down FMA onto 2^23) instead of F2I on the XU pipe.
enum { TUNE_I2FP = 1, TUNE_FMADFT = 2, TUNE_QFMA = 4, TUNE_L2PF = 8,
       TUNE_ONLY_U8 = 16,    // the launch writes uint8 rows (and accumulators) only: the other row outputs are compiled out
       TUNE_ONLY_DB = 32,    // ... f32 dB rows only
       TUNE_NO_ROWS = 64 };  // ... no rows at all (Welch / max-hold accumulators only)

// packed int16 I,Q -> float2.  Default: two I2F.S16 (XU pipe, 16 lanes/clk/SM).  TUNE_I2FP: sign-extend with
// PRMT and convert with I2FP.F32.S32 (ALU pipe) -- exact either way (|v| <= 2^15 fits a float).
template <int TUNE>
SPX_HD float2 ci16_to_f2(unsigned int w) {
#ifdef __CUDA_ARCH__
    if constexpr ((TUNE & TUNE_I2FP) != 0) {
        // prmt with the sign-replicating selector nibbles (0x8 | byte): bytes {b0, b1, sign(b1), sign(b1)} and
        // {b2, b3, sign(b3), sign(b3)}.  Inline PTX on purpose: __byte_perm() masks the selector to 3 bits per nibble.
        int lo, hi;
        asm("prmt.b32 %0, %1, 0, 0x9910;" : "=r"(lo) : "r"(w));
        asm("prmt.b32 %0, %1, 0, 0xbb32;" : "=r"(hi) : "r"(w));
        return make_float2((float)lo, (float)hi);
    }
#endif
    const short lo = (short)(w & 0xffffu), hi = (short)(w >> 16);
    return make_float2((float)lo, (float)hi);
}
template <int TUNE = 0>
SPX_HD float2 ld_stream_ci16(const short2* p) {
#ifdef __CUDA_ARCH__
    unsigned int w;
    asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(w) : "l"(p));
    return ci16_to_f2<TUNE>(w);
#else
    return make_float2((float)p->x, (float)p->y);
#endif
}
template <typename T>
SPX_HD T ld_keep(const T* p) {
#ifdef __CUDA_ARCH__
    return __ldg(p);
#else
    return *p;
#endif
}
SPX_HD float fast_sqrt(float x) {
#ifdef __CUDA_ARCH__
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return sqrtf(x);
#endif
}
SPX_HD float fast_log2(float x) {
#ifdef __CUDA_ARCH__
    float r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#else
    return log2f(x);
#endif
}
// saturating floor-convert to u8: NaN -> 0, -inf -> 0, +inf -> 255
SPX_HD unsigned int sat_floor_u8(float q) {
#ifdef __CUDA_ARCH__
    unsigned int r;
    asm("cvt.rmi.sat.u8.f32 %0, %1;" : "=r"(r) : "f"(q));
    return r;
#else
    if (!(q == q)) return 0u;
    float f = floorf(q);
    return f < 0.f ? 0u : (f > 255.f ? 255u : (unsigned int)f);
#endif
}
// The same index without the XU pipe: z = sat(y * q_a/256 + q_b/256) in [0, 1] (NaN -> 0, the scaling by 2^-8 is exact, so
// 256 z is bit-for-bit the clamped quant_pre value), z = min(z, 1 - 2^-24), then fma.rm(z, 256, 2^23) = 2^23 + floor(256 z)
// exactly: the index is the low byte of the result's bit pattern, which a byte store writes as is.
SPX_HD unsigned int sat_floor_u8_fma(float y, float q_a256, float q_b256) {
#ifdef __CUDA_ARCH__
    float z, r;
    asm("fma.rn.sat.f32 %0, %1, %2, %3;" : "=f"(z) : "f"(y), "f"(q_a256), "f"(q_b256));
    z = fminf(z, 0.99999994f);
    asm("fma.rm.f32 %0, %1, 0f43800000, 0f4B000000;" : "=f"(r) : "f"(z));
    return __float_as_uint(r);       // callers store the low byte
#else
    float z = fmaf(y, q_a256, q_b256);
    if (!(z == z) || z < 0.f) z = 0.f;
    if (z > 0.99999994f) z = 0.99999994f;
    return (unsigned int)floorf(z * 256.0f);
#endif
}
#define SPX_DB_PER_LOG2 6.02059991327962390427f  // 20*log10(2)

// dB = 20*log10(|X| + eps) (streamer.py:121) is evaluated on y = log2|X|^2: for |X|^2 >= pw_min = (2^20 eps)^2 the eps
// term changes the result by < 1e-5 dB and y = lg2(|X|^2) (one MUFU); below it y = 2 lg2(sqrt(|X|^2) + eps).
// pre-floor colormap value from y = log2|X|^2 in one FMA: (dB - vmin) * scale = q_a * y + q_b
SPX_HD float quant_pre(float y, float q_a, float q_b) {
#ifdef __CUDA_ARCH__
    return __fmaf_rn(y, q_a, q_b);
#else
    return fmaf(y, q_a, q_b);
#endif
}

// accumulator flush: Welch sum (fp64 add) and max-hold (|X|^2 >= 0, so IEEE order == unsigned order).
// `sys` selects system scope: the target may be another GPU's memory reached over NVLink, reduced into by
// several GPUs at once (the fused compute + reduction of the multi-GPU configs).
#ifdef __CUDACC__
__device__ __forceinline__ void flush_acc(double* welch, float* maxhold, long long o, float sum, float mx, int sys,
                                          double sum64 = 0.0, float mx32 = 0.f) {
    if (sys < 0) {  // system scope with a float64 addend (the final local -> peer pass)
        if (welch) atomicAdd_system(welch + o, sum64);
        if (maxhold) atomicMax_system(reinterpret_cast<unsigned int*>(maxhold) + o, __float_as_uint(mx32));
    } else if (sys) {
        if (welch) atomicAdd_system(welch + o, (double)sum);
        if (maxhold) atomicMax_system(reinterpret_cast<unsigned int*>(maxhold) + o, __float_as_uint(mx));
    } else {
        if (welch) atomicAdd(welch + o, (double)sum);
        if (maxhold) atomicMax(reinterpret_cast<unsigned int*>(maxhold) + o, __float_as_uint(mx));
    }
}
#endif

// ------------------------------------------------------------------ per-thread state
template <bool ACC>
struct StftAcc {
    float sum[ACC ? 16 : 1];
    float mx[ACC ? 16 : 1];
    SPX_HD void reset() {
#pragma unroll
        for (int i = 0; i < (ACC ? 16 : 1); ++i) { sum[i] = 0.f; mx[i] = 0.f; }
    }
};

// twiddle bases kept in registers (TW_REG): per pass s >= 1 the entries t in {1,2,3,4,8,12}
template <int N>
struct TwRegs {
    float2 b[(plan_passes(N) > 1 ? plan_passes(N) - 1 : 1) * 6];
};

template <int R> SPX_HD constexpr int tw_base_slot(int t) {
    // slot of base t in {1,2,3,4,8,12}
    return t == 1 ? 0 : t == 2 ? 1 : t == 3 ? 2 : t == 4 ? 3 : t == 8 ? 4 : 5;
}

template <int N, int S>
SPX_HD void tw_regs_load_pass(TwRegs<N>& r, int tid, const float2* tw) {
    constexpr int R = plan_radix(N, S), NS = plan_ns(N, S), OFF = plan_tw_offset(N, S);
    // only valid when the thread has one butterfly in this pass (R == 16) or all its butterflies
    // share jm (never) -- so TW_REG is restricted to plans whose passes >= 1 are all radix 16.
    static_assert(R == 16, "TW_REG needs radix-16 passes");
    const int jm = tid & (NS - 1);
    constexpr int ts[6] = {1, 2, 3, 4, 8, 12};
#pragma unroll
    for (int q = 0; q < 6; ++q) r.b[(S - 1) * 6 + q] = ld_keep(tw + OFF + (ts[q] - 1) * NS + jm);
}

// ------------------------------------------------------------------ pass pieces
template <int N, int FMT, int TUNE = 0>
SPX_HD void load_frame(float2* v, const StftParams& p, long long sample0, int tid) {
    constexpr int T = N / 16;
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        const long long i = sample0 + tid + t * T;
        if (FMT == FMT_CF32) v[t] = ld_stream_cf32(reinterpret_cast<const float2*>(p.in) + i);
        else                 v[t] = ld_stream_ci16<TUNE>(reinterpret_cast<const short2*>(p.in) + i);
    }
    if (p.win != nullptr) {
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            const float w = ld_keep(p.win + tid + t * T);
            v[t].x *= w;
            v[t].y *= w;
        }
    }
}

// pass 0 input from the shared-memory staging buffer that a bulk async copy (TMA) filled
// `win_half` is the first N/2 entries of the (symmetric) window in shared memory:
// w[i] = win_half[i] for i < N/2, win_half[N-1-i] otherwise (np.hanning / np.blackman are exactly symmetric)
template <int N, int FMT, int TUNE = 0>
SPX_HD void load_frame_staged(float2* v, const void* stage, const float* win_half, int tid) {
    constexpr int T = N / 16;
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        if (FMT == FMT_CF32) {
            v[t] = reinterpret_cast<const float2*>(stage)[tid + t * T];
        } else {
            v[t] = ci16_to_f2<TUNE>(reinterpret_cast<const unsigned int*>(stage)[tid + t * T]);
        }
    }
    if (win_half != nullptr) {
#pragma unroll
        for (int t = 0; t < 16; ++t) {
            const int i = tid + t * T;
            const float w = t < 8 ? win_half[i] : win_half[N - 1 - i];
            v[t].x *= w;
            v[t].y *= w;
        }
    }
}

template <int N, int S>
SPX_HD void pass_load_smem(float2* v, int tid, const float2* src) {
    constexpr int R = plan_radix(N, S), NB = 16 / R, T = N / 16, M = N / R;
#pragma unroll
    for (int u = 0; u < NB; ++u) {
        const int j = tid + T * u;
        // pad0(j + t*M) == pad0(j) + t*(M + M/16) because M is a multiple of 16
        const int j0 = S == 1 ? pad0(j) : j;
        constexpr int STEP = S == 1 ? M + M / 16 : M;
#pragma unroll
        for (int t = 0; t < R; ++t) v[u * R + t] = src[j0 + t * STEP];
    }
}

template <int N, int S, bool TW_IN_SMEM>
SPX_HD void pass_twiddle_table(float2* v, int tid, const float2* tw) {
    constexpr int R = plan_radix(N, S), NB = 16 / R, T = N / 16;
    constexpr int NS = plan_ns(N, S), OFF = plan_tw_offset(N, S);
#pragma unroll
    for (int u = 0; u < NB; ++u) {
        const int jm = (tid + T * u) & (NS - 1);
#pragma unroll
        for (int t = 1; t < R; ++t) {
            const float2* wp = tw + OFF + (t - 1) * NS + jm;
            v[u * R + t] = cmul(v[u * R + t], TW_IN_SMEM ? *wp : ld_keep(wp));
        }
    }
}

template <int N, int S>
SPX_HD void pass_twiddle_regs(float2* v, const TwRegs<N>& r) {
    // radix 16 only: W^{t jm}, t = 4a + b  ->  base[4a] * base[b]
    const float2* b = r.b + (S - 1) * 6;
    const float2 w1 = b[0], w2 = b[1], w3 = b[2], w4 = b[3], w8 = b[4], w12 = b[5];
    v[1] = cmul(v[1], w1);  v[2] = cmul(v[2], w2);  v[3] = cmul(v[3], w3);
    v[4] = cmul(v[4], w4);
    v[5] = cmul(v[5], cmul(w4, w1));  v[6] = cmul(v[6], cmul(w4, w2));  v[7] = cmul(v[7], cmul(w4, w3));
    v[8] = cmul(v[8], w8);
    v[9] = cmul(v[9], cmul(w8, w1));  v[10] = cmul(v[10], cmul(w8, w2)); v[11] = cmul(v[11], cmul(w8, w3));
    v[12] = cmul(v[12], w12);
    v[13] = cmul(v[13], cmul(w12, w1)); v[14] = cmul(v[14], cmul(w12, w2)); v[15] = cmul(v[15], cmul(w12, w3));
}

template <int N, int S>
SPX_HD void pass_dft(float2* v) {
    constexpr int R = plan_radix(N, S), NB = 16 / R;
#pragma unroll
    for (int u = 0; u < NB; ++u) dft<R>(v + u * R);
}

template <int N, int S>
SPX_HD void pass_store_smem(const float2* v, int tid, float2* dst) {
    constexpr int R = plan_radix(N, S), NB = 16 / R, T = N / 16, NS = plan_ns(N, S);
#pragma unroll
    for (int u = 0; u < NB; ++u) {
        const int j = tid + T * u;
        const int jm = j & (NS - 1);
        // S == 0: i = 16 j + t  ->  pad0(i) = 17 j + t
        const int base = S == 0 ? 17 * j : (j - jm) * R + jm;
#pragma unroll
        for (int t = 0; t < R; ++t) dst[base + t * NS] = v[u * R + t];
    }
}

// bin held in v[u*R + t] after the last pass
template <int N>
SPX_HD int out_bin(int tid, int u, int t) {
    constexpr int S = plan_passes(N) - 1, R = plan_radix(N, S), T = N / 16;
    return tid + T * u + t * (N / R);
}

// ------------------------------------------------------------------ fused epilogue
// row position (fftshift order, streamer.py:119) of v[u*R + t]:  ((bin + N/2) mod N)
//   = shift_off(t) + tid + T*u   because N/2 is a multiple of N/R and tid + T*u < N/R
template <int N>
SPX_HD constexpr int shift_off(int t) {
    constexpr int S = plan_passes(N) - 1, R = plan_radix(N, S);
    return (t * (N / R) + N / 2) & (N - 1);
}

template <int N, bool ACC, int TUNE = 0>
SPX_HD void epilogue(float2* v, int tid, const StftParams& p, long long row, StftAcc<ACC>& acc) {
    constexpr int S = plan_passes(N) - 1, R = plan_radix(N, S), NB = 16 / R, T = N / 16;
    // which row outputs exist: read from the parameters, or fixed at compile time for the launcher's specialised instantiations
    constexpr bool FIXED = (TUNE & (TUNE_ONLY_U8 | TUNE_ONLY_DB | TUNE_NO_ROWS)) != 0;
    const bool want_spec = FIXED ? false : p.spec_rows != nullptr;
    const bool want_db = FIXED ? (TUNE & TUNE_ONLY_DB) != 0 : p.db_rows != nullptr;
    const bool want_wf = FIXED ? (TUNE & TUNE_ONLY_U8) != 0 : p.wf_rows != nullptr;
    if (want_spec) {
        float2* sp = p.spec_rows + row * N + tid;
#pragma unroll
        for (int u = 0; u < NB; ++u)
#pragma unroll
            for (int t = 0; t < R; ++t) sp[shift_off<N>(t) + T * u] = v[u * R + t];
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i].x = v[i].x * v[i].x + v[i].y * v[i].y;  // |X|^2
    if (ACC) {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            acc.sum[i] += v[i].x;
            acc.mx[i] = fmaxf(acc.mx[i], v[i].x);
        }
    }
    if (want_db || want_wf) {
        // smallest of this thread's 16 powers decides (one branch) whether the eps term can matter
        float m01 = fminf(v[0].x, v[1].x), m23 = fminf(v[2].x, v[3].x), m45 = fminf(v[4].x, v[5].x);
        float m67 = fminf(v[6].x, v[7].x), m89 = fminf(v[8].x, v[9].x), mab = fminf(v[10].x, v[11].x);
        float mcd = fminf(v[12].x, v[13].x), mef = fminf(v[14].x, v[15].x);
        const float pmin = fminf(fminf(fminf(m01, m23), fminf(m45, m67)), fminf(fminf(m89, mab), fminf(mcd, mef)));
        // v[i].y = log2 of the (eps-corrected) power: dB = (10 log10 2) * y
        if (pmin >= p.db_pw_min) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i].y = fast_log2(v[i].x);
        } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i].y = 2.0f * fast_log2(fast_sqrt(v[i].x) + p.db_eps);
        }
        if (want_db) {
            float* db = p.db_rows + row * N + tid;
#pragma unroll
            for (int u = 0; u < NB; ++u)
#pragma unroll
                for (int t = 0; t < R; ++t) db[shift_off<N>(t) + T * u] = (0.5f * SPX_DB_PER_LOG2) * v[u * R + t].y;
        }
        if (want_wf) {
            unsigned char* wf = p.wf_rows + row * N + tid;
            if constexpr ((TUNE & TUNE_QFMA) != 0) {
                const float qa = p.q_a * 0.00390625f, qb = p.q_b * 0.00390625f;
#pragma unroll
                for (int u = 0; u < NB; ++u)
#pragma unroll
                    for (int t = 0; t < R; ++t)
                        wf[shift_off<N>(t) + T * u] = (unsigned char)sat_floor_u8_fma(v[u * R + t].y, qa, qb);
            } else {
#pragma unroll
                for (int u = 0; u < NB; ++u)
#pragma unroll
                    for (int t = 0; t < R; ++t)
                        wf[shift_off<N>(t) + T * u] = (unsigned char)sat_floor_u8(quant_pre(v[u * R + t].y, p.q_a, p.q_b));
            }
        }
    }
}

// what a flush writes: (slot position, value) pairs are produced by the caller with atomics
template <int N>
SPX_HD int acc_pos(int tid, int idx) {
    constexpr int S = plan_passes(N) - 1, R = plan_radix(N, S), T = N / 16;
    return shift_off<N>(idx % R) + tid + T * (idx / R);
}

// ------------------------------------------------------------------ one frame, phase by phase
// phase k (0 <= k < P) = pass k; barriers between phases are the caller's job.
template <int N, int FMT, bool ACC, int TWM, int S, int TUNE = 0>
SPX_HD void stft_phase(float2* v, int tid, const StftParams& p, long long sample0, long long row, bool active,
                       float2* bufA, float2* bufB, const float2* tw, const TwRegs<N>& twr, StftAcc<ACC>& acc,
                       const void* stage = nullptr, const float* win_half = nullptr) {
    constexpr int P = plan_passes(N);
    if (!active) return;
    if constexpr (S == 0) {
        if (stage) load_frame_staged<N, FMT, TUNE>(v, stage, win_half, tid);
        else load_frame<N, FMT, TUNE>(v, p, sample0, tid);
    } else {
        const float2* src = ((S - 1) & 1) ? bufB : bufA;
        pass_load_smem<N, S>(v, tid, src);
        if constexpr (TWM == TW_REG) pass_twiddle_regs<N, S>(v, twr);
        else pass_twiddle_table<N, S, TWM == TW_SMEM>(v, tid, tw);
    }
    pass_dft<N, S>(v);
    if constexpr (S == P - 1) {
        epilogue<N, ACC>(v, tid, p, row, acc);
    } else {
        float2* dst = (S & 1) ? bufB : bufA;
        pass_store_smem<N, S>(v, tid, dst);
    }
}

}  // namespace spx
