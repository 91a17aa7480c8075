// spx_plan.h -- the opaque plan object behind include/spx.h, and the per-device state of the plan-less calls (host-side only).
#pragma once
#include <cuda_runtime.h>

#include <initializer_list>
#include <map>
#include <mutex>
#include <vector>

#include "spx_internal.h"

namespace spx {

struct DevBuf {
    void* ptr = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes);  // grow-only
    void release();
};

// What the plan-less one-shot calls (spx_classify_features, spx_iq_hist2d, spx_frame_stats, spx_stream_frame_f64) keep per
// device.  Each call holds `mu` while it uses the context, so the calls on one device serialise.
struct DeviceCtx {
    std::mutex mu;
    cudaStream_t st = nullptr;   // non-blocking: every host-memory call, and the device-memory calls of the histogram, frame
                                 // stats and features without a caller stream (spx_stream_frame_f64 keeps the caller's)
    int sm_count = 0;
    DevBuf stage;                // device staging of host-memory calls (grow-only)
    cudaMemPool_t hist_pool = nullptr;   // spx_iq_hist2d's per-CTA tables (stream-ordered: calls on other streams may overlap)
    std::map<int, double2*> tw64;        // spx_stream_frame_f64: n -> device table of n/2 float64 twiddles
    // Reserves `stage` for parts of these sizes, each at a 256-byte aligned offset, and points part[i] at part i.
    int carve(std::initializer_list<size_t> bytes, void** part);
};

// The context of `device` (0 <= device < min(device count, 64)), made current, with its stream and SM count set up.
int device_ctx(int device, DeviceCtx** out);

}  // namespace spx

struct spx_plan {
    spx_plan_config cfg{};
    int sm_count = 0;
    float* d_win = nullptr;   // window * in_scale (nullptr: rect and scale 1)
    float2* d_tw = nullptr;   // twiddle table of the shared-memory kernel (nfft <= 8192)
    std::vector<double> win64;
    double sum_w2 = 0.0, sum_w = 0.0;
    cudaStream_t s_compute = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    // the ingest ring uploads consecutive slots on alternating streams (s_h2d, s_h2d_alt): two uploads in flight keep the H2D
    // direction full while the D2H direction is busy -- a single copy at a time leaves ~35 us per 16 MB slot on the table
    // (tools/micro/copy_gap.cu: 386 vs 355 us per slot; needs >= 5 slots in flight in the ring to show, profiles/r02_e2e_ring_depth.jsonl)
    cudaStream_t s_h2d_alt = nullptr;
    std::vector<cudaEvent_t> events;
    size_t piece_bytes = 16u << 20;  // H2D piece size of the host pipeline
    size_t peer_piece_bytes = 48u << 20;  // uint8 rows per piece of the peer-output pipeline (two staging buffers)
    size_t persist_rows_bytes = 64u << 20;  // uint8 row buffer of a device-resident persistence call without caller rows
    size_t pool_rows_bytes = 256u << 20;    // float dB row buffer of a pooled call without caller dB rows (measured, DESIGN.md K8)
    // staging for SPX_MEM_HOST execution (grow-only)
    spx::DevBuf st_in, st_db, st_wf, st_spec, st_welch, st_max, st_misc, st_flush;
    // persistence spectrum / pooled spectrogram: counts or pooled accumulator staging of the host path, and the plan-owned
    // row buffer (uint8 levels or float dB rows; device path without caller rows; host path without caller rows, one piece)
    spx::DevBuf st_sink, st_rows;
    // large-N (four-step) path, nfft >= 16384
    int big_n1 = 0, big_n2 = 0;
    float2* d_big_tw = nullptr;  // one allocation holding the four tables below
    float2 *d_tw1 = nullptr, *d_tw2 = nullptr, *d_wn_fine = nullptr, *d_wn_coarse = nullptr;
    size_t big_scratch_bytes = 384u << 20;  // two halves of 192 MB: frames per batch = half / (nfft * 8); measured best on B200
    spx::DevBuf st_big;
    float2* d_big2 = nullptr;      // K2v2 (single-kernel 65536-point path): N = 4096 twiddle table followed by the base table
    size_t big2_tw_count = 0;
    float* d_big2_win = nullptr;   // K2v2 window table in phase A's thread order
    cudaStream_t s_big_aux = nullptr;             // column kernels of batch k+1 run here, next to the row kernels of batch k
    cudaEvent_t ev_big[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // entry, A done x2, B done x2
    // Bluestein path (nfft not a power of two, or < 16): inner power-of-two plan of length blu_m
    int blu_m = 0;
    spx_plan* blu_inner = nullptr;
    float2* d_blu = nullptr;  // [N] window*scale*chirp, [N] chirp/M, [M] FFT_M(conj chirp) in fftshift order
    // ordering of plan-owned scratch between calls on different streams
    cudaEvent_t ev_scratch = nullptr;
    cudaStream_t scratch_stream = nullptr;
    bool scratch_stream_valid = false;
    std::mutex mu;
};

namespace spx {
// *out = events[i], creating events up to i on demand
int event_at(std::vector<cudaEvent_t>& events, size_t i, cudaEvent_t* out);
// Plan-owned scratch (K2 halves, the K2v2 scratch and its counters, the Bluestein buffers) is shared by every call on the
// plan, whatever stream it runs on.  A call that uses it brackets its kernels on `st`: scratch_wait makes `st` wait for
// the last such call if that one ran on another stream, scratch_record marks `st` as the stream now using it.
bool plan_has_scratch(const spx_plan* pl);
int scratch_wait(spx_plan* pl, cudaStream_t st);
int scratch_record(spx_plan* pl, cudaStream_t st);

// Outputs of an STFT launch, in device memory: rows [r][N] (dB, uint8 levels, spectrum) and accumulators [s][N] (Welch
// sums, max-hold).  A null member is not produced.  vmin / vmax set the uint8 levels; sys_atomics makes the accumulator
// flushes system-scope (accumulators on another GPU).
struct StftOut {
    float* db = nullptr;
    unsigned char* wf = nullptr;
    float2* spec = nullptr;
    double* welch = nullptr;
    float* maxhold = nullptr;
    float vmin = 0.f, vmax = 1.f;
    int sys_atomics = 0;
    bool has_rows() const { return db || wf || spec; }
    // the rows from row r0 on, or the accumulators of stream s, of rows of N bins; null members stay null
    StftOut rows_at(size_t r0, size_t N) const {
        StftOut o = *this;
        if (db) o.db = db + r0 * N;
        if (wf) o.wf = wf + r0 * N;
        if (spec) o.spec = spec + r0 * N;
        return o;
    }
    StftOut stream_at(long long s, size_t N) const {
        StftOut o = *this;
        if (welch) o.welch = welch + (size_t)s * N;
        if (maxhold) o.maxhold = maxhold + (size_t)s * N;
        return o;
    }
    // the row epilogue's uint8 level = q_a * log2(power) + q_b
    float q_a() const { return (float)(3.01029995663981195214 * 256.0 / ((double)vmax - (double)vmin)); }  // 10 log10(2) * scale
    float q_b() const { return (float)(-(double)vmin * 256.0 / ((double)vmax - (double)vmin)); }
};
// the row epilogue's power floor, (2^20 eps)^2
inline float db_pw_min(const spx_plan* pl) { return pl->cfg.db_eps * pl->cfg.db_eps * 1099511627776.0f; }

int stft_launch_device(spx_plan* pl, const void* in, long long n_streams, long long stream_stride, long long frames,
                       const StftOut& out, cudaStream_t st);
int bigfft_plan_init(spx_plan* pl);
int bigfft_launch_stream(spx_plan* pl, const void* in, long long frames, long long row0, const StftOut& out, cudaStream_t st);
int peer_reduce_launch(const double* w_local, const float* m_local, double* w_peer, float* m_peer, long long n, cudaStream_t st);
int big2_plan_init(spx_plan* pl);
bool big2_eligible(const spx_plan* pl, const void* in, const StftOut& out);
int big2_launch_stream(spx_plan* pl, const void* in, long long frames, long long row0, const StftOut& out, cudaStream_t st);
int persist_launch(const spx_plan* pl, const uint8_t* rows, long long n_streams, long long frames, uint32_t* counts,
                   cudaStream_t st);
// a pooled call (spx_pool_args, checked)
struct PoolCall {
    int mode;
    long long frames_per_row;
    int bins_per_col;
    long long first_frame, n_rows;
};
// rows [n_streams][frames][nfft] into acc [n_streams][n_rows][nfft / bins_per_col]; frame0: global index of frame 0
int pool_launch(const spx_plan* pl, const float* rows, long long n_streams, long long frames, long long frame0,
                const PoolCall& pc, double* acc, cudaStream_t st);
int pool_fill_launch(double* acc, long long n, int mode, cudaStream_t st);
int pool_finalize_launch(const spx_plan* pl, const double* acc, long long n_streams, long long G, long long F_total,
                         long long K, int B, int mode, float vmin, float vmax, float* db_out, uint8_t* wf_out,
                         cudaStream_t st);
int welch_finalize_launch(const double* acc, int n, double inv_norm, double* pxx, double* pxx_db, cudaStream_t st);
int bluestein_plan_init(spx_plan* pl);
int bluestein_launch_stream(spx_plan* pl, const void* in, long long frames, long long row0, const StftOut& out,
                            cudaStream_t st);
}  // namespace spx
