// spx_api.cu -- the C ABI of libspx (include/spx.h): plans, device/host execution, staging.
//
// Host-memory execution (SPX_MEM_HOST) is a three-stream pipeline: pieces of the input go
// host->device on `s_h2d`, every piece releases the frames it completes to the fused kernel on
// `s_compute`, and finished rows drain device->host on `s_d2h`; all three overlap when the
// caller's buffers are pinned (spx_host_alloc / spx_host_register).  This is the new
// "pinned, double-buffered" ingest of SURVEY.md section 0 (the reference queues one dict per
// rx buffer: /root/reference/app/sdr/streamer.py:123-131,186-194).
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <new>
#include <vector>

#include <nvtx3/nvToolsExt.h>

#include "spx_plan.h"
#include "spx_pool_device.cuh"
#include "spx_stft_kernel.cuh"
#include "spx_tables.h"

namespace spx {

static thread_local char g_err[512] = "";

NvtxRange::NvtxRange(const char* name) { nvtxRangePushA(name); }
NvtxRange::~NvtxRange() { nvtxRangePop(); }

int spx_set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

static bool is_pow2(long long v) { return v > 0 && (v & (v - 1)) == 0; }

int DevBuf::reserve(size_t bytes) {
    if (bytes <= cap) return SPX_OK;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&ptr, want);
    if (e != cudaSuccess) {
        ptr = nullptr;
        return spx_set_error(SPX_E_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    }
    cap = want;
    return SPX_OK;
}
void DevBuf::release() {
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
}

struct KernelOnDevice {
    const void* kern;
    int dev;
    bool operator<(const KernelOnDevice& o) const { return kern != o.kern ? kern < o.kern : dev < o.dev; }
};

int kernel_setup(const void* kern, int threads, size_t smem, int* occ) {
    static std::mutex mu;
    static std::map<KernelOnDevice, int> occ_of;   // blocks per SM
    int dev = 0;
    SPX_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> g(mu);
    const KernelOnDevice key{kern, dev};
    auto it = occ_of.find(key);
    if (it == occ_of.end()) {
        int o = 0;
        SPX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SPX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, threads, smem));
        it = occ_of.emplace(key, o).first;
    }
    if (occ) *occ = it->second;
    return SPX_OK;
}

int DeviceCtx::carve(std::initializer_list<size_t> bytes, void** part) {
    size_t total = 0;
    for (size_t b : bytes) total += (b + 255) & ~(size_t)255;
    SPX_TRY(stage.reserve(total));
    char* p = (char*)stage.ptr;
    for (size_t b : bytes) {
        *part++ = p;
        p += (b + 255) & ~(size_t)255;
    }
    return SPX_OK;
}

int check_device(int device) {
    int ndev = 0;
    SPX_TRY(spx_device_count(&ndev));
    if (ndev == 0) return spx_set_error(SPX_E_NODEVICE, "no CUDA device (libspx has no CPU fallback)");
    if (device < 0 || device >= ndev) return spx_set_error(SPX_E_INVALID, "device %d out of range (%d devices)", device, ndev);
    SPX_CUDA(cudaSetDevice(device));
    return SPX_OK;
}

size_t env_bytes(const char* name, size_t fallback, long long min) {
    const char* e = getenv(name);
    const long long v = e ? atoll(e) : 0;
    return v >= min ? (size_t)v : fallback;
}

int device_ctx(int device, DeviceCtx** out) {
    static DeviceCtx ctx[64];
    SPX_TRY(check_device(device));
    if (device >= 64) return spx_set_error(SPX_E_INVALID, "device %d: at most 64 devices", device);
    DeviceCtx& c = ctx[device];
    std::lock_guard<std::mutex> g(c.mu);
    if (!c.st) {
        SPX_CUDA(cudaDeviceGetAttribute(&c.sm_count, cudaDevAttrMultiProcessorCount, device));
        SPX_CUDA(cudaStreamCreateWithFlags(&c.st, cudaStreamNonBlocking));
    }
    *out = &c;
    return SPX_OK;
}

int event_at(std::vector<cudaEvent_t>& events, size_t i, cudaEvent_t* out) {
    while (events.size() <= i) {
        cudaEvent_t e;
        SPX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        events.push_back(e);
    }
    *out = events[i];
    return SPX_OK;
}

// ------------------------------------------------------------------ plan-owned scratch across streams
bool plan_has_scratch(const spx_plan* pl) { return pl->cfg.nfft > 8192 || pl->blu_m != 0; }

int scratch_wait(spx_plan* pl, cudaStream_t st) {
    if (!pl->ev_scratch) SPX_CUDA(cudaEventCreateWithFlags(&pl->ev_scratch, cudaEventDisableTiming));
    if (pl->scratch_stream_valid && pl->scratch_stream != st) SPX_CUDA(cudaStreamWaitEvent(st, pl->ev_scratch, 0));
    return SPX_OK;
}

int scratch_record(spx_plan* pl, cudaStream_t st) {
    SPX_CUDA(cudaEventRecord(pl->ev_scratch, st));
    pl->scratch_stream = st;
    pl->scratch_stream_valid = true;
    return SPX_OK;
}

// ------------------------------------------------------------------ dispatch
static size_t in_elt(const spx_plan* pl) { return pl->cfg.in_fmt == SPX_FMT_CI16 ? 4 : 8; }

int stft_launch_device(spx_plan* pl, const void* in, long long n_streams, long long stream_stride, long long frames,
                       const StftOut& out, cudaStream_t st) {
    if (frames <= 0 || n_streams <= 0) return SPX_OK;
    // arbitrary length (Bluestein over the inner power-of-two plan) and the four-step path: one stream at a time
    if (pl->blu_m || pl->cfg.nfft >= 16384) {
        const auto launch_stream = pl->blu_m ? bluestein_launch_stream : bigfft_launch_stream;
        for (long long s = 0; s < n_streams; ++s)
            SPX_TRY(launch_stream(pl, (const char*)in + (size_t)(s * stream_stride) * in_elt(pl), frames, s * frames,
                                  out.stream_at(s, pl->cfg.nfft), st));
        return SPX_OK;
    }
    StftLaunch L;
    memset(&L, 0, sizeof(L));
    L.p.in = in;
    L.p.stream_stride = stream_stride;
    L.p.frames_per_stream = frames;
    L.p.n_streams = (int)n_streams;
    L.p.hop = pl->cfg.hop;
    L.p.win = pl->d_win;
    L.p.tw = pl->d_tw;
    L.p.db_rows = out.db;
    L.p.wf_rows = out.wf;
    L.p.spec_rows = out.spec;
    L.p.welch_acc = out.welch;
    L.p.maxhold = out.maxhold;
    L.p.db_eps = pl->cfg.db_eps;
    L.p.db_pw_min = db_pw_min(pl);
    L.p.sys_atomics = out.sys_atomics;
    L.p.q_a = out.q_a();
    L.p.q_b = out.q_b();
    L.nfft = pl->cfg.nfft;
    L.in_fmt = pl->cfg.in_fmt;
    L.variant = pl->cfg.variant;
    L.sm_count = pl->sm_count;
    L.total_frames = frames * n_streams;
    L.stream = st;
    const int n = pl->cfg.nfft;
    if (n <= 512) return launch_stft_small(L);
    if (n <= 2048) return launch_stft_1k2k(L);
    if (n == 4096) return launch_stft_4k(L);
    if (n == 8192) return launch_stft_8k(L);
    return spx_set_error(SPX_E_UNSUPPORTED, "nfft %d: large-N path not built yet", n);
}

// ------------------------------------------------------------------ row consumers
// The persistence spectrum consumes uint8 rows and the pooled spectrogram float dB rows.  Without caller rows of that kind
// the STFT of frames [0, F) of every stream goes in batches through the plan's row buffer (SPX_PERSIST_ROWS_BYTES of
// uint8 rows, or SPX_POOL_ROWS_BYTES of float rows), each batch followed by its consumer kernel on the same stream, so
// those rows never leave the GPU.  The buffer holds max(1, bytes / (S row)) frames of the S streams of a batch: it
// exceeds its size only when a single frame of every stream does.  A batch starts f0 * hop samples into every stream:
// f0 * hop * elt keeps the input alignment (128 bytes for K1v2, 16 bytes for K1's staged loads and K2v2) and K2v2's
// hop % 256 of the unbatched call, and a batch covers all streams with the call's stride, so each batch runs the kernel
// family the unbatched call would.  Exception: caller rows of several streams must land at rows s * F + f, so those
// batches run one stream at a time.
enum RowKind { ROWS_U8, ROWS_DB };

// The consumer of a call's rows besides the caller, if `acc` is set: the persistence counts [S][256][N] (uint32) of the
// uint8 levels, or, when `pool` is set, the pooled accumulator [S][n_rows][N / B] (float64) of the float dB rows.  `acc`
// is stream 0's accumulator, in the call's memory space or in device staging.
struct RowSink {
    char* acc = nullptr;
    const PoolCall* pool = nullptr;
    RowKind kind() const { return pool ? ROWS_DB : ROWS_U8; }
    size_t stream_bytes(int N) const {
        return pool ? (size_t)(pool->n_rows * (N / pool->bins_per_col)) * sizeof(double) : (size_t)256 * N * sizeof(uint32_t);
    }
    RowSink stream_at(long long s, int N) const {
        RowSink k = *this;
        if (acc) k.acc = acc + (size_t)s * stream_bytes(N);
        return k;
    }
    // the rows of `out` this sink reads (null: none)
    const void* rows_of(const StftOut& out) const { return pool ? (const void*)out.db : (const void*)out.wf; }
    // over rows [S][F][N] of streams 0 .. S - 1 here, whose frame 0 is frame f0 of the call
    int launch(const spx_plan* pl, const void* rows, long long S, long long F, long long f0, cudaStream_t st) const {
        if (pool) return pool_launch(pl, (const float*)rows, S, F, pool->first_frame + f0, *pool, (double*)acc, st);
        return persist_launch(pl, (const uint8_t*)rows, S, F, (uint32_t*)acc, st);
    }
};

static size_t row_bytes(const spx_plan* pl, RowKind kind) { return (size_t)pl->cfg.nfft * (kind == ROWS_DB ? sizeof(float) : 1); }

static long long row_batch_frames(const spx_plan* pl, RowKind kind, long long Sb, long long F) {
    long long fb = (long long)((kind == ROWS_DB ? pl->pool_rows_bytes : pl->persist_rows_bytes) / ((size_t)Sb * row_bytes(pl, kind)));
    if (fb < 1) fb = 1;
    return fb < F ? fb : F;
}

// The STFT of frames [0, F) of S streams into `out`, then `sink` over their rows: the caller's rows when `out` has rows
// of the sink's kind, else batches through the row buffer.  f0: the call's index of frame 0 here.
static int stft_then_sink(spx_plan* pl, const char* in, long long S, long long stride, long long F, long long f0,
                          const StftOut& out, const RowSink& sink, cudaStream_t st) {
    if (!sink.acc || sink.rows_of(out)) {
        SPX_TRY(stft_launch_device(pl, in, S, stride, F, out, st));
        return sink.acc ? sink.launch(pl, sink.rows_of(out), S, F, f0, st) : SPX_OK;
    }
    const int N = pl->cfg.nfft, hop = pl->cfg.hop;
    const RowKind kind = sink.kind();
    const long long Sb = S > 1 && out.has_rows() ? 1 : S;
    const long long fb = row_batch_frames(pl, kind, Sb, F);
    SPX_TRY(pl->st_rows.reserve((size_t)(Sb * fb) * row_bytes(pl, kind)));   // a no-op when the host pipeline reserved it up front
    void* rows = pl->st_rows.ptr;
    for (long long s = 0; s < S; s += Sb) {
        for (long long b0 = 0; b0 < F; b0 += fb) {
            const long long nf = F - b0 < fb ? F - b0 : fb;
            StftOut o = out.rows_at((size_t)(s * F + b0), N).stream_at(s, N);
            if (kind == ROWS_DB) o.db = (float*)rows;
            else o.wf = (unsigned char*)rows;
            SPX_TRY(stft_launch_device(pl, in + (size_t)(s * stride + b0 * hop) * in_elt(pl), Sb, stride, nf, o, st));
            SPX_TRY(sink.stream_at(s, N).launch(pl, rows, Sb, nf, f0 + b0, st));
        }
    }
    return SPX_OK;
}

// The accumulators of a call in the caller's memory, in staging order: Welch sums, max-hold, the sink's.  Without
// `accumulate` they start from zero, a pooled accumulator from the identity of pool->mode; `stage` is the device staging
// of a host-memory call.
struct CallAcc {
    void* ptr;
    size_t bytes;
    const PoolCall* pool;
    DevBuf* stage;
};

static std::vector<CallAcc> call_accs(spx_plan* pl, const spx_stft_args* a, const RowSink& sink) {
    const size_t S = (size_t)a->n_streams;
    const int N = pl->cfg.nfft;
    std::vector<CallAcc> v;
    if (a->welch_acc) v.push_back({a->welch_acc, S * N * sizeof(double), nullptr, &pl->st_welch});
    if (a->maxhold) v.push_back({a->maxhold, S * N * sizeof(float), nullptr, &pl->st_max});
    if (sink.acc) v.push_back({sink.acc, S * sink.stream_bytes(N), sink.pool, &pl->st_sink});
    return v;
}

static int reset_on_device(const CallAcc& c, void* acc, cudaStream_t st) {
    if (c.pool) return pool_fill_launch((double*)acc, (long long)(c.bytes / sizeof(double)), c.pool->mode, st);
    SPX_CUDA(cudaMemsetAsync(acc, 0, c.bytes, st));
    return SPX_OK;
}

// ------------------------------------------------------------------ host-memory pipeline
static int stft_exec_host(spx_plan* pl, spx_stft_args* a, long long F, const RowSink& sink) {
    const int N = pl->cfg.nfft, hop = pl->cfg.hop;
    const size_t elt = in_elt(pl);
    const long long S = a->n_streams, L = a->n_samples;
    const long long stride_host = S > 1 ? a->stream_stride : 0;
    const size_t rows = (size_t)(S * F);
    const std::vector<CallAcc> accs = call_accs(pl, a, sink);
    SPX_TRY(pl->st_in.reserve((size_t)(S * L) * elt));
    if (a->db_rows) SPX_TRY(pl->st_db.reserve(rows * N * sizeof(float)));
    if (a->wf_rows) SPX_TRY(pl->st_wf.reserve(rows * N));
    if (a->spec_rows) SPX_TRY(pl->st_spec.reserve(rows * N * sizeof(float2)));
    for (const CallAcc& c : accs) SPX_TRY(c.stage->reserve(c.bytes));
    char* d_in = (char*)pl->st_in.ptr;
    StftOut d_out;   // the outputs in device staging
    d_out.db = a->db_rows ? (float*)pl->st_db.ptr : nullptr;
    d_out.wf = a->wf_rows ? (unsigned char*)pl->st_wf.ptr : nullptr;
    d_out.spec = a->spec_rows ? (float2*)pl->st_spec.ptr : nullptr;
    d_out.welch = a->welch_acc ? (double*)pl->st_welch.ptr : nullptr;
    d_out.maxhold = a->maxhold ? (float*)pl->st_max.ptr : nullptr;
    d_out.vmin = a->vmin;
    d_out.vmax = a->vmax;
    RowSink d_sink = sink;
    if (sink.acc) d_sink.acc = (char*)pl->st_sink.ptr;
    long long h2d = 0, d2h = 0;

    // plan-owned scratch (four-step / K2v2 / Bluestein buffers, the row buffer): a device-resident call on a caller stream
    // may still be using it, so the kernels queued here on s_compute wait for that call first, as the device path does
    const bool own_rows = sink.acc && !sink.rows_of(d_out);
    const bool owns_scratch = plan_has_scratch(pl) || own_rows;
    if (owns_scratch) SPX_TRY(scratch_wait(pl, pl->s_compute));

    // accumulators: start from the caller's running values or from their reset value
    for (const CallAcc& c : accs) {
        if (a->accumulate) {
            SPX_CUDA(cudaMemcpyAsync(c.stage->ptr, c.ptr, c.bytes, cudaMemcpyHostToDevice, pl->s_compute));
            h2d += (long long)c.bytes;
        } else {
            SPX_TRY(reset_on_device(c, c.stage->ptr, pl->s_compute));
        }
    }

    // piece size: big enough to amortise launches, small enough to overlap (about 8-16 MiB)
    long long piece = (long long)(pl->piece_bytes / elt);
    if (piece < (long long)N * 4) piece = (long long)N * 4;
    // a sink without rows: one row buffer for every piece, sized for the largest (a piece spans at most `piece` samples, so
    // at most piece / hop + 1 frames), reserved here -- growing it between pieces would free device memory, which
    // synchronises the device in the middle of the pipeline
    if (own_rows) {
        const long long most = piece / hop + 2 < F ? piece / hop + 2 : F;
        SPX_TRY(pl->st_rows.reserve((size_t)row_batch_frames(pl, sink.kind(), 1, most) * row_bytes(pl, sink.kind())));
    }
    struct Piece { long long s, f_lo, f_hi; };
    std::vector<Piece> pieces;
    size_t ev = 0;
    for (long long s = 0; s < S; ++s) {
        const char* h_in = (const char*)a->in + (size_t)(s * stride_host) * elt;
        char* dd = d_in + (size_t)(s * L) * elt;
        long long f_lo = 0;
        // piece schedule: ramp up from piece/8 and back down at the end, so that the un-overlapped head (first H2D
        // before any kernel) and tail (last D2H after the last kernel) of the three-stream pipeline stay short
        long long step = 0;
        int k = 0;
        for (long long lo = 0; lo < L; lo += step, ++k) {
            const long long left = L - lo;
            step = piece >> (k < 3 ? 3 - k : 0);
            if (left <= piece) step = left > piece / 4 ? (left + 1) / 2 : left;
            if (step < (long long)N) step = (long long)N;
            const long long hi = lo + step < L ? lo + step : L;
            // (one upload stream here: alternating the pieces over s_h2d / s_h2d_alt as the ingest ring does was measured
            // slower for this fully pre-queued pipeline -- 8.3 vs 10.2 GS/s on config 2)
            {
                NvtxRange r("spx H2D piece");
                SPX_CUDA(cudaMemcpyAsync(dd + (size_t)lo * elt, h_in + (size_t)lo * elt, (size_t)(hi - lo) * elt,
                                         cudaMemcpyHostToDevice, pl->s_h2d));
            }
            h2d += (hi - lo) * (long long)elt;
            long long f_hi = spx_frame_count(hi, N, hop);
            if (hi == L) f_hi = F;
            if (f_hi <= f_lo) continue;
            cudaEvent_t e_in, e_k;
            SPX_TRY(event_at(pl->events, ev++, &e_in));
            SPX_TRY(event_at(pl->events, ev++, &e_k));
            SPX_CUDA(cudaEventRecord(e_in, pl->s_h2d));
            SPX_CUDA(cudaStreamWaitEvent(pl->s_compute, e_in, 0));
            NvtxRange r_k("spx STFT kernel piece");
            SPX_TRY(stft_then_sink(pl, dd + (size_t)(f_lo * hop) * elt, 1, 0, f_hi - f_lo, f_lo,
                                   d_out.rows_at((size_t)(s * F + f_lo), N).stream_at(s, N), d_sink.stream_at(s, N),
                                   pl->s_compute));
            SPX_CUDA(cudaEventRecord(e_k, pl->s_compute));
            pieces.push_back({s, f_lo, f_hi});
            f_lo = f_hi;
        }
    }
    // drain rows as their kernels finish
    NvtxRange r_d2h("spx D2H rows");
    size_t evi = 1;
    for (const Piece& pc : pieces) {
        cudaEvent_t e_k = pl->events[evi];
        evi += 2;
        if (!d_out.has_rows()) continue;
        SPX_CUDA(cudaStreamWaitEvent(pl->s_d2h, e_k, 0));
        const size_t r0 = (size_t)(pc.s * F + pc.f_lo), nr = (size_t)(pc.f_hi - pc.f_lo);
        if (d_out.db) {
            SPX_CUDA(cudaMemcpyAsync(a->db_rows + r0 * N, d_out.db + r0 * N, nr * N * sizeof(float), cudaMemcpyDeviceToHost, pl->s_d2h));
            d2h += (long long)(nr * N * sizeof(float));
        }
        if (d_out.wf) {
            SPX_CUDA(cudaMemcpyAsync(a->wf_rows + r0 * N, d_out.wf + r0 * N, nr * N, cudaMemcpyDeviceToHost, pl->s_d2h));
            d2h += (long long)(nr * N);
        }
        if (d_out.spec) {
            SPX_CUDA(cudaMemcpyAsync(a->spec_rows + r0 * N * 2, d_out.spec + r0 * N, nr * N * sizeof(float2), cudaMemcpyDeviceToHost, pl->s_d2h));
            d2h += (long long)(nr * N * sizeof(float2));
        }
    }
    for (const CallAcc& c : accs) {
        SPX_CUDA(cudaMemcpyAsync(c.ptr, c.stage->ptr, c.bytes, cudaMemcpyDeviceToHost, pl->s_compute));
        d2h += (long long)c.bytes;
    }
    if (owns_scratch) SPX_TRY(scratch_record(pl, pl->s_compute));
    SPX_CUDA(cudaStreamSynchronize(pl->s_h2d));
    SPX_CUDA(cudaStreamSynchronize(pl->s_h2d_alt));
    SPX_CUDA(cudaStreamSynchronize(pl->s_compute));
    SPX_CUDA(cudaStreamSynchronize(pl->s_d2h));
    a->h2d_bytes_out = h2d;
    a->d2h_bytes_out = d2h;
    return SPX_OK;
}

// ------------------------------------------------------------------ device execution with peer-resident outputs
// Multi-GPU capture shards (SURVEY.md 8(e)): the accumulators and the waterfall rows live on another GPU.
// The Welch / max-hold partials are reduced by the STFT kernel itself (system-scope atomics over NVLink, tiny
// traffic).  The uint8 rows are produced in frame pieces into two local staging buffers and pushed to the peer by
// the copy engine on `s_d2h` while the next piece is being transformed: full-size NVLink writes instead of the
// kernel's 16..32-byte row fragments, and the transfer hides behind the transform piece by piece.
// last hop of the hierarchical reduction (registers -> this GPU's L2 -> the owner's HBM over NVLink)
__global__ void peer_reduce_kernel(const double* __restrict__ w_local, const float* __restrict__ m_local, double* w_peer,
                                   float* m_peer, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        flush_acc(w_local ? w_peer : nullptr, m_local ? m_peer : nullptr, i, 0.f, 0.f, -1, w_local ? w_local[i] : 0.0,
                  m_local ? m_local[i] : 0.f);
}

int peer_reduce_launch(const double* w_local, const float* m_local, double* w_peer, float* m_peer, long long n, cudaStream_t st) {
    if (n <= 0 || (!w_local && !m_local)) return SPX_OK;
    peer_reduce_kernel<<<(unsigned)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184), 256, 0, st>>>(w_local, m_local, w_peer, m_peer, n);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

static int stft_exec_device_peer(spx_plan* pl, spx_stft_args* a, long long F, cudaStream_t st) {
    const int N = pl->cfg.nfft, hop = pl->cfg.hop;
    const size_t elt = in_elt(pl);
    const long long S = a->n_streams;
    // partials accumulate in local memory (device-scope atomics in L2); one system-scope pass at the end adds them
    // to the owner's buffers: S*N remote atomics per call instead of one per chunk flush
    double* w_local = nullptr;
    float* m_local = nullptr;
    if (a->welch_acc) {
        SPX_TRY(pl->st_welch.reserve((size_t)S * N * sizeof(double)));
        w_local = (double*)pl->st_welch.ptr;
        SPX_CUDA(cudaMemsetAsync(w_local, 0, (size_t)S * N * sizeof(double), st));
    }
    if (a->maxhold) {
        SPX_TRY(pl->st_max.reserve((size_t)S * N * sizeof(float)));
        m_local = (float*)pl->st_max.ptr;
        SPX_CUDA(cudaMemsetAsync(m_local, 0, (size_t)S * N * sizeof(float), st));
    }
    long long piece = (long long)(pl->peer_piece_bytes / (size_t)N);
    if (piece < 1) piece = 1;
    if (piece > F) piece = F;
    // rows that live on THIS GPU (the owner's own shard, peer_outputs bit 1 clear) are written by the kernel
    // directly: no staging, no copy
    const bool rows_local = (a->peer_outputs & 2) == 0;
    unsigned char* stage[2] = {nullptr, nullptr};
    if (a->wf_rows && !rows_local) {
        SPX_TRY(pl->st_wf.reserve((size_t)(2 * piece) * N));
        stage[0] = (unsigned char*)pl->st_wf.ptr;
        stage[1] = stage[0] + (size_t)piece * N;
    } else {
        piece = F;  // nothing to stage: one launch per stream
    }
    cudaEvent_t e_k[2], e_c[2];
    for (int i = 0; i < 2; ++i) {
        SPX_TRY(event_at(pl->events, (size_t)i, &e_k[i]));
        SPX_TRY(event_at(pl->events, (size_t)(2 + i), &e_c[i]));
    }
    const StftOut local{nullptr, a->wf_rows, nullptr, w_local, m_local, a->vmin, a->vmax};
    long long idx = 0;
    for (long long s = 0; s < S; ++s) {
        const char* in_s = (const char*)a->in + (size_t)(s * a->stream_stride) * elt;
        for (long long f_lo = 0; f_lo < F; f_lo += piece, ++idx) {
            const long long nf = F - f_lo < piece ? F - f_lo : piece;
            const int b = (int)(idx & 1);
            const bool staged = a->wf_rows && !rows_local;
            if (idx >= 2 && staged) SPX_CUDA(cudaStreamWaitEvent(st, e_c[b], 0));   // the copy that last used this buffer is done
            StftOut o = local.rows_at((size_t)(s * F + f_lo), N).stream_at(s, N);
            if (staged) o.wf = stage[b];
            SPX_TRY(stft_launch_device(pl, in_s + (size_t)(f_lo * hop) * elt, 1, 0, nf, o, st));
            if (!staged) continue;
            SPX_CUDA(cudaEventRecord(e_k[b], st));
            SPX_CUDA(cudaStreamWaitEvent(pl->s_d2h, e_k[b], 0));
            SPX_CUDA(cudaMemcpyAsync(a->wf_rows + (size_t)(s * F + f_lo) * N, stage[b], (size_t)nf * N, cudaMemcpyDefault, pl->s_d2h));
            SPX_CUDA(cudaEventRecord(e_c[b], pl->s_d2h));
        }
    }
    if (w_local || m_local) {
        NvtxRange r("spx peer reduce (system-scope atomics over NVLink)");
        SPX_TRY(peer_reduce_launch(w_local, m_local, a->welch_acc, a->maxhold, S * N, st));
    }
    // whoever waits on `st` (spx_plan_sync, a later launch) also waits for the last copies
    if (a->wf_rows && !rows_local) {
        SPX_CUDA(cudaStreamWaitEvent(st, e_c[0], 0));
        if (idx >= 2) SPX_CUDA(cudaStreamWaitEvent(st, e_c[1], 0));
    }
    a->d2h_bytes_out = 0;
    return SPX_OK;
}

__global__ void __launch_bounds__(256) fp32_probe_kernel(float* out, int iters, float a, float b) {
    float r[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) r[i] = threadIdx.x * 1e-3f + (float)i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 16; ++i) r[i] = fmaf(r[i], a, b);
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += r[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// L2 flush for measurements: READ a buffer twice the L2 size (clean lines replace the cache contents; a write-flush
// would leave dirty lines whose write-back then competes with the timed kernel)
__global__ void __launch_bounds__(256) l2_flush_read_kernel(const uint4* __restrict__ buf, size_t n_vec, unsigned int* sink) {
    unsigned int acc = 0u;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n_vec; i += (size_t)gridDim.x * blockDim.x) {
        const uint4 v = buf[i];
        acc ^= v.x ^ v.y ^ v.z ^ v.w;
    }
    if (acc == 0x9e3779b9u) *sink = acc;   // never true for a zeroed buffer; keeps the loads alive
}

__global__ void welch_finalize_kernel(const double* __restrict__ acc, int n, double inv_norm, double* pxx, double* pxx_db) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = acc[i] * inv_norm;
    if (pxx) pxx[i] = v;
    if (pxx_db) pxx_db[i] = 10.0 * log10(v);
}

int welch_finalize_launch(const double* acc, int n, double inv_norm, double* pxx, double* pxx_db, cudaStream_t st) {
    welch_finalize_kernel<<<(n + 255) / 256, 256, 0, st>>>(acc, n, inv_norm, pxx, pxx_db);
    SPX_CUDA(cudaGetLastError());
    return SPX_OK;
}

}  // namespace spx

using namespace spx;

// =================================================================== extern "C"
extern "C" {

int spx_abi_version(void) { return SPX_ABI_VERSION; }
const char* spx_last_error(void) { return g_err; }

int spx_device_count(int* count) {
    if (!count) return spx_set_error(SPX_E_INVALID, "count is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *count = 0;
        return spx_set_error(SPX_E_NODEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *count = n;
    return SPX_OK;
}

int spx_get_device_info(int device, spx_device_info* out) {
    if (!out) return spx_set_error(SPX_E_INVALID, "out is NULL");
    cudaDeviceProp pr;
    SPX_CUDA(cudaGetDeviceProperties(&pr, device));
    memset(out, 0, sizeof(*out));
    out->struct_size = sizeof(*out);
    out->sm_count = pr.multiProcessorCount;
    out->cc_major = pr.major;
    out->cc_minor = pr.minor;
    out->l2_bytes = pr.l2CacheSize;
    out->max_smem_optin = (int)pr.sharedMemPerBlockOptin;
    out->total_mem = (int64_t)pr.totalGlobalMem;
    strncpy(out->name, pr.name, sizeof(out->name) - 1);
    return SPX_OK;
}

int64_t spx_frame_count(int64_t n_samples, int32_t nfft, int32_t hop) {
    if (nfft <= 0 || hop <= 0 || n_samples < nfft) return 0;
    return (n_samples - nfft) / hop + 1;
}

int spx_host_alloc(void** out, size_t bytes) {
    if (!out) return spx_set_error(SPX_E_INVALID, "out is NULL");
    SPX_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
    return SPX_OK;
}
int spx_host_alloc_wc(void** out, size_t bytes) {
    if (!out) return spx_set_error(SPX_E_INVALID, "out is NULL");
    SPX_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable | cudaHostAllocWriteCombined));
    return SPX_OK;
}
int spx_host_free(void* p) {
    if (p) SPX_CUDA(cudaFreeHost(p));
    return SPX_OK;
}
int spx_host_register(void* p, size_t bytes) {
    SPX_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return SPX_OK;
}
int spx_host_unregister(void* p) {
    SPX_CUDA(cudaHostUnregister(p));
    return SPX_OK;
}

int spx_device_alloc(int device, void** out, size_t bytes) {
    if (!out) return spx_set_error(SPX_E_INVALID, "out is NULL");
    SPX_CUDA(cudaSetDevice(device));
    cudaError_t e = cudaMalloc(out, bytes ? bytes : 1);
    if (e != cudaSuccess) return spx_set_error(SPX_E_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    return SPX_OK;
}
int spx_device_free(int device, void* p) {
    SPX_CUDA(cudaSetDevice(device));
    if (p) SPX_CUDA(cudaFree(p));
    return SPX_OK;
}
int spx_memcpy_h2d(int device, void* dst, const void* src, size_t bytes) {
    SPX_CUDA(cudaSetDevice(device));
    SPX_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
    return SPX_OK;
}
int spx_memcpy_d2h(int device, void* dst, const void* src, size_t bytes) {
    SPX_CUDA(cudaSetDevice(device));
    SPX_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
    return SPX_OK;
}
int spx_memcpy_d2h_async(int device, void* dst_host, const void* src, size_t bytes, void* stream) {
    SPX_CUDA(cudaSetDevice(device));
    SPX_CUDA(cudaMemcpyAsync(dst_host, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return SPX_OK;
}
int spx_memset(int device, void* dst, int value, size_t bytes) {
    SPX_CUDA(cudaSetDevice(device));
    SPX_CUDA(cudaMemset(dst, value, bytes));
    return SPX_OK;
}
int spx_device_sync(int device) {
    SPX_CUDA(cudaSetDevice(device));
    SPX_CUDA(cudaDeviceSynchronize());
    return SPX_OK;
}

int spx_ipc_export(int device, void* dptr, void* handle_out) {
    if (!dptr || !handle_out) return spx_set_error(SPX_E_INVALID, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == SPX_IPC_HANDLE_BYTES, "handle size");
    SPX_CUDA(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    SPX_CUDA(cudaIpcGetMemHandle(&h, dptr));
    memcpy(handle_out, &h, sizeof(h));
    return SPX_OK;
}
int spx_ipc_open(int device, const void* handle, void** dptr_out) {
    if (!handle || !dptr_out) return spx_set_error(SPX_E_INVALID, "NULL argument");
    SPX_CUDA(cudaSetDevice(device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    SPX_CUDA(cudaIpcOpenMemHandle(dptr_out, h, cudaIpcMemLazyEnablePeerAccess));
    return SPX_OK;
}
int spx_ipc_close(int device, void* dptr) {
    if (!dptr) return SPX_OK;
    SPX_CUDA(cudaSetDevice(device));
    SPX_CUDA(cudaIpcCloseMemHandle(dptr));
    return SPX_OK;
}

int spx_plan_create(spx_plan** out, const spx_plan_config* cfg) {
    if (!out || !cfg) return spx_set_error(SPX_E_INVALID, "NULL argument");
    *out = nullptr;
    if (cfg->struct_size != sizeof(spx_plan_config))
        return spx_set_error(SPX_E_INVALID, "spx_plan_config.struct_size %u != %zu", cfg->struct_size, sizeof(spx_plan_config));
    const bool native_len = is_pow2(cfg->nfft) && cfg->nfft >= 16;
    if (cfg->nfft < 1 || cfg->nfft > (1 << 20) || (!native_len && cfg->nfft > (1 << 19)))
        return spx_set_error(SPX_E_UNSUPPORTED, "nfft %d: supported lengths are powers of two in [16, 1048576] and any length in [1, 524288]", cfg->nfft);
    if (cfg->hop < 1 || cfg->hop > cfg->nfft) return spx_set_error(SPX_E_INVALID, "hop %d must be in [1, nfft]", cfg->hop);
    if (cfg->window < 0 || cfg->window > 2) return spx_set_error(SPX_E_INVALID, "unknown window %d", cfg->window);
    if (cfg->in_fmt != SPX_FMT_CF32 && cfg->in_fmt != SPX_FMT_CI16) return spx_set_error(SPX_E_INVALID, "unknown in_fmt %d", cfg->in_fmt);
    if (cfg->variant != 0 && cfg->variant != 1 && cfg->variant != 12 && cfg->variant != 22)
        return spx_set_error(SPX_E_INVALID, "unknown variant %d: accepted values are 0, 1, 12 and 22 (see spx.h)", cfg->variant);
    SPX_TRY(check_device(cfg->device));

    spx_plan* pl = new (std::nothrow) spx_plan();
    if (!pl) return spx_set_error(SPX_E_NOMEM, "out of host memory");
    pl->cfg = *cfg;
    if (!(pl->cfg.in_scale != 0.0f)) pl->cfg.in_scale = 1.0f;
    pl->peer_piece_bytes = env_bytes("SPX_PEER_PIECE_BYTES", pl->peer_piece_bytes, 4096);
    pl->piece_bytes = env_bytes("SPX_H2D_PIECE_BYTES", pl->piece_bytes, 65536);
    pl->big_scratch_bytes = env_bytes("SPX_BIG_SCRATCH_BYTES", pl->big_scratch_bytes, 1 << 20);
    // the row buffers hold at least one row
    pl->persist_rows_bytes = std::max(env_bytes("SPX_PERSIST_ROWS_BYTES", pl->persist_rows_bytes, 1), (size_t)cfg->nfft);
    pl->pool_rows_bytes = std::max(env_bytes("SPX_POOL_ROWS_BYTES", pl->pool_rows_bytes, 1), (size_t)cfg->nfft * sizeof(float));
    int rc = SPX_OK;
    do {
        cudaError_t e;
        if ((e = cudaDeviceGetAttribute(&pl->sm_count, cudaDevAttrMultiProcessorCount, cfg->device)) != cudaSuccess) { rc = spx_set_error(SPX_E_CUDA, "%s", cudaGetErrorString(e)); break; }
        // window (float64 as numpy builds it, scaled, rounded once to float)
        pl->win64 = build_window_f64(cfg->window, cfg->nfft);
        pl->sum_w2 = 0.0;
        pl->sum_w = 0.0;
        for (double w : pl->win64) { pl->sum_w2 += w * w; pl->sum_w += w; }
        if (cfg->window != SPX_WINDOW_RECT || pl->cfg.in_scale != 1.0f) {
            std::vector<float> wf((size_t)cfg->nfft);
            for (int i = 0; i < cfg->nfft; ++i) wf[i] = (float)(pl->win64[i] * (double)pl->cfg.in_scale);
            if ((e = cudaMalloc(&pl->d_win, wf.size() * sizeof(float))) != cudaSuccess) { rc = spx_set_error(SPX_E_NOMEM, "%s", cudaGetErrorString(e)); break; }
            if ((e = cudaMemcpy(pl->d_win, wf.data(), wf.size() * sizeof(float), cudaMemcpyHostToDevice)) != cudaSuccess) { rc = spx_set_error(SPX_E_CUDA, "%s", cudaGetErrorString(e)); break; }
        }
        if (!native_len) {
            if ((rc = bluestein_plan_init(pl)) != SPX_OK) break;
        } else if (cfg->nfft > 8192) {
            if ((rc = bigfft_plan_init(pl)) != SPX_OK) break;
            if ((rc = big2_plan_init(pl)) != SPX_OK) break;
        } else {
            std::vector<float2> tw = build_twiddles(cfg->nfft);
            if ((e = cudaMalloc(&pl->d_tw, tw.size() * sizeof(float2))) != cudaSuccess) { rc = spx_set_error(SPX_E_NOMEM, "%s", cudaGetErrorString(e)); break; }
            if ((e = cudaMemcpy(pl->d_tw, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice)) != cudaSuccess) { rc = spx_set_error(SPX_E_CUDA, "%s", cudaGetErrorString(e)); break; }
        }
        if ((e = cudaStreamCreateWithFlags(&pl->s_compute, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&pl->s_h2d, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&pl->s_h2d_alt, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&pl->s_d2h, cudaStreamNonBlocking)) != cudaSuccess) { rc = spx_set_error(SPX_E_CUDA, "%s", cudaGetErrorString(e)); break; }
    } while (0);
    if (rc != SPX_OK) {
        spx_plan_destroy(pl);
        return rc;
    }
    *out = pl;
    return SPX_OK;
}

int spx_plan_destroy(spx_plan* pl) {
    if (!pl) return SPX_OK;
    cudaSetDevice(pl->cfg.device);
    if (pl->s_compute) { cudaStreamSynchronize(pl->s_compute); cudaStreamDestroy(pl->s_compute); }
    if (pl->s_h2d) { cudaStreamSynchronize(pl->s_h2d); cudaStreamDestroy(pl->s_h2d); }
    if (pl->s_h2d_alt) { cudaStreamSynchronize(pl->s_h2d_alt); cudaStreamDestroy(pl->s_h2d_alt); }
    if (pl->s_d2h) { cudaStreamSynchronize(pl->s_d2h); cudaStreamDestroy(pl->s_d2h); }
    for (cudaEvent_t e : pl->events) cudaEventDestroy(e);
    if (pl->d_win) cudaFree(pl->d_win);
    if (pl->d_tw) cudaFree(pl->d_tw);
    if (pl->s_big_aux) { cudaStreamSynchronize(pl->s_big_aux); cudaStreamDestroy(pl->s_big_aux); }
    for (cudaEvent_t e : pl->ev_big) if (e) cudaEventDestroy(e);
    if (pl->d_big_tw) cudaFree(pl->d_big_tw);
    if (pl->ev_scratch) cudaEventDestroy(pl->ev_scratch);
    if (pl->d_big2) cudaFree(pl->d_big2);
    if (pl->d_big2_win) cudaFree(pl->d_big2_win);
    if (pl->d_blu) cudaFree(pl->d_blu);
    if (pl->blu_inner) spx_plan_destroy(pl->blu_inner);
    pl->st_big.release();
    pl->st_in.release(); pl->st_db.release(); pl->st_wf.release(); pl->st_spec.release();
    pl->st_welch.release(); pl->st_max.release(); pl->st_misc.release(); pl->st_flush.release();
    pl->st_sink.release(); pl->st_rows.release();
    delete pl;
    return SPX_OK;
}

int spx_plan_sync(spx_plan* pl) {
    if (!pl) return spx_set_error(SPX_E_INVALID, "plan is NULL");
    std::lock_guard<std::mutex> g(pl->mu);
    SPX_CUDA(cudaSetDevice(pl->cfg.device));
    SPX_CUDA(cudaStreamSynchronize(pl->s_h2d));
    SPX_CUDA(cudaStreamSynchronize(pl->s_h2d_alt));
    SPX_CUDA(cudaStreamSynchronize(pl->s_compute));
    SPX_CUDA(cudaStreamSynchronize(pl->s_d2h));
    return SPX_OK;
}

int spx_fp32_peak(int device, double* tflops_out) {
    if (!tflops_out) return spx_set_error(SPX_E_INVALID, "tflops_out is NULL");
    SPX_CUDA(cudaSetDevice(device));
    int sm = 0;
    SPX_CUDA(cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, device));
    const int blocks = sm * 8, iters = 1 << 13;
    float* out = nullptr;
    SPX_CUDA(cudaMalloc(&out, sizeof(float) * (size_t)blocks * 256));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    float best = 1e30f;
    for (int k = 0; k < 6; ++k) {
        cudaEventRecord(e0, 0);
        fp32_probe_kernel<<<blocks, 256>>>(out, iters, 1.0001f, 0.5f);
        cudaEventRecord(e1, 0);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        if (k > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaError_t e = cudaGetLastError();
    cudaFree(out);
    if (e != cudaSuccess) return spx_set_error(SPX_E_CUDA, "fp32 probe: %s", cudaGetErrorString(e));
    *tflops_out = 2.0 * (double)blocks * 256.0 * (double)iters * 16.0 / ((double)best * 1e-3) / 1e12;
    return SPX_OK;
}

int spx_plan_stream(spx_plan* pl, void** stream_out) {
    if (!pl || !stream_out) return spx_set_error(SPX_E_INVALID, "NULL argument");
    *stream_out = (void*)pl->s_compute;
    return SPX_OK;
}

struct spx_timer {
    int device;
    cudaEvent_t e0, e1;
};

int spx_timer_create(int32_t device, spx_timer** out) {
    if (!out) return spx_set_error(SPX_E_INVALID, "out is NULL");
    *out = nullptr;
    SPX_CUDA(cudaSetDevice(device));
    spx_timer* t = new (std::nothrow) spx_timer();
    if (!t) return spx_set_error(SPX_E_NOMEM, "out of host memory");
    t->device = device;
    cudaError_t e = cudaEventCreate(&t->e0);
    if (e == cudaSuccess) e = cudaEventCreate(&t->e1);
    if (e != cudaSuccess) {
        delete t;
        return spx_set_error(SPX_E_CUDA, "cudaEventCreate: %s", cudaGetErrorString(e));
    }
    *out = t;
    return SPX_OK;
}
int spx_timer_start(spx_timer* t, void* stream) {
    if (!t) return spx_set_error(SPX_E_INVALID, "timer is NULL");
    SPX_CUDA(cudaSetDevice(t->device));
    SPX_CUDA(cudaEventRecord(t->e0, (cudaStream_t)stream));
    return SPX_OK;
}
int spx_timer_stop(spx_timer* t, void* stream) {
    if (!t) return spx_set_error(SPX_E_INVALID, "timer is NULL");
    SPX_CUDA(cudaSetDevice(t->device));
    SPX_CUDA(cudaEventRecord(t->e1, (cudaStream_t)stream));
    return SPX_OK;
}
int spx_timer_elapsed_ms(spx_timer* t, float* ms_out) {
    if (!t || !ms_out) return spx_set_error(SPX_E_INVALID, "NULL argument");
    SPX_CUDA(cudaSetDevice(t->device));
    SPX_CUDA(cudaEventSynchronize(t->e1));
    SPX_CUDA(cudaEventElapsedTime(ms_out, t->e0, t->e1));
    return SPX_OK;
}
int spx_timer_destroy(spx_timer* t) {
    if (!t) return SPX_OK;
    cudaSetDevice(t->device);
    cudaEventDestroy(t->e0);
    cudaEventDestroy(t->e1);
    delete t;
    return SPX_OK;
}

int spx_plan_window_sums(spx_plan* pl, double* sum_w2, double* sum_w) {
    if (!pl) return spx_set_error(SPX_E_INVALID, "plan is NULL");
    if (sum_w2) *sum_w2 = pl->sum_w2;  // window only: in_scale belongs to the data
    if (sum_w) *sum_w = pl->sum_w;
    return SPX_OK;
}

// spx_stft_exec, plus `sink` over the call's rows when sink.acc is not NULL
static int stft_exec(spx_plan* pl, spx_stft_args* a, const RowSink& sink) {
    if (!pl || !a) return spx_set_error(SPX_E_INVALID, "NULL argument");
    if (a->struct_size != sizeof(spx_stft_args))
        return spx_set_error(SPX_E_INVALID, "spx_stft_args.struct_size %u != %zu", a->struct_size, sizeof(spx_stft_args));
    if (sink.acc && a->peer_outputs)
        return spx_set_error(SPX_E_UNSUPPORTED, "%s with peer_outputs is not supported", sink.pool ? "pooling" : "persistence");
    if (a->n_streams < 1) return spx_set_error(SPX_E_INVALID, "n_streams must be >= 1");
    if (a->n_samples < 0) return spx_set_error(SPX_E_INVALID, "n_samples < 0");
    if (a->mem != SPX_MEM_HOST && a->mem != SPX_MEM_DEVICE) return spx_set_error(SPX_E_INVALID, "unknown mem %d", a->mem);
    if ((a->wf_rows != nullptr) && !(a->vmax > a->vmin)) return spx_set_error(SPX_E_INVALID, "wf_rows needs vmax > vmin");
    if (sink.acc && sink.kind() == ROWS_U8 && !(a->vmax > a->vmin))
        return spx_set_error(SPX_E_INVALID, "persistence needs vmax > vmin");
    if (a->n_streams > 1 && a->stream_stride < a->n_samples && a->mem == SPX_MEM_HOST)
        return spx_set_error(SPX_E_INVALID, "stream_stride < n_samples");
    const long long F = spx_frame_count(a->n_samples, pl->cfg.nfft, pl->cfg.hop);
    const PoolCall* pc = sink.pool;
    if (pc && F > 0 && pool_row_of(pc->first_frame + F - 1, pc->frames_per_row) >= pc->n_rows)
        return spx_set_error(SPX_E_INVALID, "frames %lld .. %lld fall outside the %lld pooled rows of %lld frames",
                             pc->first_frame, pc->first_frame + F - 1, pc->n_rows, pc->frames_per_row);
    a->n_frames_out = F;
    a->h2d_bytes_out = 0;
    a->d2h_bytes_out = 0;
    std::lock_guard<std::mutex> g(pl->mu);
    SPX_CUDA(cudaSetDevice(pl->cfg.device));
    if (a->in == nullptr && F > 0) return spx_set_error(SPX_E_INVALID, "in is NULL");
    if (a->mem == SPX_MEM_DEVICE) {
        cudaStream_t st = a->stream ? (cudaStream_t)a->stream : pl->s_compute;
        const StftOut out{a->db_rows, a->wf_rows, reinterpret_cast<float2*>(a->spec_rows), a->welch_acc, a->maxhold,
                          a->vmin, a->vmax, a->peer_outputs ? 1 : 0};
        // Plan-owned scratch (four-step / K2v2 scratch and counters, Bluestein buffers, peer staging, the row buffer) is
        // shared by every call on this plan: a call on another stream than the previous one waits for that one's kernels
        // first.
        const bool owns_scratch = plan_has_scratch(pl) || a->peer_outputs || (sink.acc && !sink.rows_of(out));
        if (owns_scratch) SPX_TRY(scratch_wait(pl, st));
        if (!a->accumulate)
            for (const CallAcc& c : call_accs(pl, a, sink)) SPX_TRY(reset_on_device(c, c.ptr, st));
        int rc;
        if (a->peer_outputs && !a->db_rows && !a->spec_rows && F > 0) rc = stft_exec_device_peer(pl, a, F, st);
        else rc = stft_then_sink(pl, (const char*)a->in, a->n_streams, a->stream_stride, F, 0, out, sink, st);
        if (rc == SPX_OK && owns_scratch) rc = scratch_record(pl, st);
        return rc;
    }
    if (F == 0) {   // nothing to run: the accumulators are reset in host memory
        if (!a->accumulate)
            for (const CallAcc& c : call_accs(pl, a, sink)) {
                if (c.pool) std::fill_n((double*)c.ptr, c.bytes / sizeof(double), c.pool->mode == SPX_POOL_MAX ? -INFINITY : 0.0);
                else memset(c.ptr, 0, c.bytes);
            }
        return SPX_OK;
    }
    return stft_exec_host(pl, a, F, sink);
}

int spx_stft_exec(spx_plan* pl, spx_stft_args* a) { return stft_exec(pl, a, RowSink{}); }

int spx_stft_exec_persistence(spx_plan* pl, spx_stft_args* a, uint32_t* counts) {
    if (!counts) return spx_set_error(SPX_E_INVALID, "counts is NULL");
    return stft_exec(pl, a, RowSink{(char*)counts, nullptr});
}

// K, B and the mode of a pooled call or its finalisation
static int check_pool_shape(const spx_plan* pl, int mode, long long K, int B) {
    if (mode != SPX_POOL_MEAN && mode != SPX_POOL_MAX) return spx_set_error(SPX_E_INVALID, "unknown pool mode %d", mode);
    if (K < 1) return spx_set_error(SPX_E_INVALID, "frames_per_row %lld must be >= 1", K);
    if (B < 1 || pl->cfg.nfft % B != 0)
        return spx_set_error(SPX_E_INVALID, "bins_per_col %d must be >= 1 and divide nfft %d", B, pl->cfg.nfft);
    return SPX_OK;
}

int spx_stft_exec_pooled(spx_plan* pl, spx_stft_args* a, spx_pool_args* p) {
    if (!pl || !a || !p) return spx_set_error(SPX_E_INVALID, "NULL argument");
    if (p->struct_size != sizeof(spx_pool_args))
        return spx_set_error(SPX_E_INVALID, "spx_pool_args.struct_size %u != %zu", p->struct_size, sizeof(spx_pool_args));
    SPX_TRY(check_pool_shape(pl, p->mode, p->frames_per_row, p->bins_per_col));
    if (p->first_frame < 0 || p->n_rows < 0) return spx_set_error(SPX_E_INVALID, "first_frame and n_rows must be >= 0");
    if (!p->acc) return spx_set_error(SPX_E_INVALID, "acc is NULL");
    const PoolCall pc{p->mode, p->frames_per_row, p->bins_per_col, p->first_frame, p->n_rows};
    return stft_exec(pl, a, RowSink{(char*)p->acc, &pc});
}

int spx_pool_finalize(spx_plan* pl, int32_t mem, int32_t mode, const double* acc, int32_t n_streams, int64_t n_rows,
                      int64_t n_frames_total, int64_t frames_per_row, int32_t bins_per_col, float* db_out, uint8_t* wf_out,
                      float vmin, float vmax, void* stream) {
    if (!pl || !acc) return spx_set_error(SPX_E_INVALID, "NULL argument");
    SPX_TRY(check_pool_shape(pl, mode, frames_per_row, bins_per_col));
    if (mem != SPX_MEM_HOST && mem != SPX_MEM_DEVICE) return spx_set_error(SPX_E_INVALID, "unknown mem %d", mem);
    if (n_streams < 1 || n_frames_total < 0) return spx_set_error(SPX_E_INVALID, "n_streams must be >= 1, n_frames_total >= 0");
    if (n_rows != (n_frames_total + frames_per_row - 1) / frames_per_row)
        return spx_set_error(SPX_E_INVALID, "n_rows %lld != ceil(%lld frames / %lld)", (long long)n_rows,
                             (long long)n_frames_total, (long long)frames_per_row);
    if (wf_out && !(vmax > vmin)) return spx_set_error(SPX_E_INVALID, "wf_out needs vmax > vmin");
    std::lock_guard<std::mutex> g(pl->mu);
    SPX_CUDA(cudaSetDevice(pl->cfg.device));
    const size_t n = (size_t)n_streams * (size_t)n_rows * (size_t)(pl->cfg.nfft / bins_per_col);
    if (mem == SPX_MEM_DEVICE) {
        cudaStream_t st = stream ? (cudaStream_t)stream : pl->s_compute;
        return pool_finalize_launch(pl, acc, n_streams, n_rows, n_frames_total, frames_per_row, bins_per_col, mode, vmin,
                                    vmax, db_out, wf_out, st);
    }
    if (n == 0 || (!db_out && !wf_out)) return SPX_OK;
    // host memory: [acc | dB | levels] staged in one buffer
    SPX_TRY(pl->st_misc.reserve(n * (sizeof(double) + sizeof(float) + 1)));
    double* d_acc = (double*)pl->st_misc.ptr;
    float* d_db = (float*)(d_acc + n);
    uint8_t* d_wf = (uint8_t*)(d_db + n);
    SPX_CUDA(cudaMemcpyAsync(d_acc, acc, n * sizeof(double), cudaMemcpyHostToDevice, pl->s_compute));
    SPX_TRY(pool_finalize_launch(pl, d_acc, n_streams, n_rows, n_frames_total, frames_per_row, bins_per_col, mode, vmin, vmax,
                                 db_out ? d_db : nullptr, wf_out ? d_wf : nullptr, pl->s_compute));
    if (db_out) SPX_CUDA(cudaMemcpyAsync(db_out, d_db, n * sizeof(float), cudaMemcpyDeviceToHost, pl->s_compute));
    if (wf_out) SPX_CUDA(cudaMemcpyAsync(wf_out, d_wf, n, cudaMemcpyDeviceToHost, pl->s_compute));
    SPX_CUDA(cudaStreamSynchronize(pl->s_compute));
    return SPX_OK;
}

int spx_stft_time(spx_plan* pl, spx_stft_args* a, int32_t warmup, int32_t iters, int32_t flush_l2, float* ms_each) {
    if (!pl || !a || !ms_each || iters < 1 || warmup < 0) return spx_set_error(SPX_E_INVALID, "bad argument");
    if (a->mem != SPX_MEM_DEVICE) return spx_set_error(SPX_E_INVALID, "spx_stft_time needs SPX_MEM_DEVICE buffers");
    cudaEvent_t e0, e1;
    size_t flush_bytes = 256u << 20;
    {
        std::lock_guard<std::mutex> g(pl->mu);
        SPX_CUDA(cudaSetDevice(pl->cfg.device));
        if (flush_l2 && pl->st_flush.cap < flush_bytes + 256) {
            SPX_TRY(pl->st_flush.reserve(flush_bytes + 256));
            SPX_CUDA(cudaMemset(pl->st_flush.ptr, 0, flush_bytes + 256));
        }
    }
    SPX_CUDA(cudaEventCreate(&e0));
    SPX_CUDA(cudaEventCreate(&e1));
    cudaStream_t st = a->stream ? (cudaStream_t)a->stream : pl->s_compute;
    int rc = SPX_OK;
    for (int i = 0; i < warmup + iters && rc == SPX_OK; ++i) {
        if (flush_l2)
            l2_flush_read_kernel<<<pl->sm_count * 8, 256, 0, st>>>((const uint4*)pl->st_flush.ptr, flush_bytes / 16,
                                                                   (unsigned int*)((char*)pl->st_flush.ptr + flush_bytes));
        cudaEventRecord(e0, st);
        rc = spx_stft_exec(pl, a);
        cudaEventRecord(e1, st);
        cudaError_t e = cudaEventSynchronize(e1);
        if (rc == SPX_OK && e != cudaSuccess) rc = spx_set_error(SPX_E_CUDA, "kernel failed: %s", cudaGetErrorString(e));
        if (rc == SPX_OK && i >= warmup) cudaEventElapsedTime(&ms_each[i - warmup], e0, e1);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return rc;
}

int spx_welch_finalize(spx_plan* pl, int32_t mem, const double* welch_acc, int64_t n_frames, double fs, double* pxx,
                       double* pxx_db, void* stream) {
    return spx_welch_finalize_batch(pl, mem, welch_acc, 1, n_frames, fs, pxx, pxx_db, stream);
}

int spx_welch_finalize_batch(spx_plan* pl, int32_t mem, const double* welch_acc, int32_t n_streams, int64_t n_frames,
                             double fs, double* pxx, double* pxx_db, void* stream) {
    if (!pl || !welch_acc) return spx_set_error(SPX_E_INVALID, "NULL argument");
    if (n_frames < 1 || !(fs > 0) || n_streams < 1) return spx_set_error(SPX_E_INVALID, "n_frames, fs and n_streams must be positive");
    std::lock_guard<std::mutex> g(pl->mu);
    SPX_CUDA(cudaSetDevice(pl->cfg.device));
    const int N = pl->cfg.nfft * n_streams;  // element-wise: the batch is one long array
    // mlab.psd: |X|^2 / (Fs * sum(w^2)), mean over frames.  in_scale is part of the data, not of the window.
    const double inv = 1.0 / ((double)n_frames * fs * pl->sum_w2);
    if (mem == SPX_MEM_DEVICE) {
        cudaStream_t st = stream ? (cudaStream_t)stream : pl->s_compute;
        welch_finalize_kernel<<<(N + 255) / 256, 256, 0, st>>>(welch_acc, N, inv, pxx, pxx_db);
        SPX_CUDA(cudaGetLastError());
        return SPX_OK;
    }
    SPX_TRY(pl->st_misc.reserve((size_t)N * sizeof(double) * 3));
    double* d = (double*)pl->st_misc.ptr;
    SPX_CUDA(cudaMemcpyAsync(d, welch_acc, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, pl->s_compute));
    welch_finalize_kernel<<<(N + 255) / 256, 256, 0, pl->s_compute>>>(d, N, inv, pxx ? d + N : nullptr, pxx_db ? d + 2 * N : nullptr);
    SPX_CUDA(cudaGetLastError());
    if (pxx) SPX_CUDA(cudaMemcpyAsync(pxx, d + N, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, pl->s_compute));
    if (pxx_db) SPX_CUDA(cudaMemcpyAsync(pxx_db, d + 2 * N, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, pl->s_compute));
    SPX_CUDA(cudaStreamSynchronize(pl->s_compute));
    return SPX_OK;
}

}  // extern "C"
