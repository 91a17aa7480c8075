// spx_ring.cu -- pinned host ring buffer with multi-buffered async ingest (north_star: "app/sdr gains a
// pinned host ring buffer with double-buffered cudaMemcpyAsync, and H2D bytes are reported separately").
//
// Replaces the reference's frame queue of per-buffer dicts (/root/reference/app/sdr/streamer.py:18,
// 123-131,186-200): the producer writes raw samples straight into a page-locked slot, commit() enqueues
// H2D (copy stream) -> fused STFT kernel (compute stream) -> D2H of the slot's results (drain stream),
// and returns immediately; the next slot can be filled while the previous ones are in flight.
// The stream is continuous across slots: the (N - hop)-sample tail that the next frames still need is
// carried device-to-device into the head of the next slot's device buffer, never re-sent over PCIe.
#include <string.h>

#include <stdio.h>
#include <stdlib.h>

#include <mutex>
#include <new>
#include <vector>

#include "spx_plan.h"

namespace spx {

struct RingSlot {
    void* h_in = nullptr;            // pinned, slot_samples * elt
    char* d_in = nullptr;            // device, (nfft + slot_samples) * elt : [carry][new samples]
    unsigned char *d_wf = nullptr, *h_wf = nullptr;
    float *d_db = nullptr, *h_db = nullptr;
    double *d_welch = nullptr, *h_welch = nullptr;
    float *d_max = nullptr, *h_max = nullptr;
    double *d_pdb = nullptr, *h_pdb = nullptr;       // Welch PSD of the slot in dB (want_features)
    spx_features *d_feat = nullptr, *h_feat = nullptr;
    // Welch sum, PSD in dB, max-hold and the feature record live in ONE device block and ONE pinned block ([welch][pdb][max][feat]):
    // a slot's small results leave in a single copy -- as four copies they held the D2H queue ~40 us per 350 us slot
    char *d_small = nullptr, *h_small = nullptr;
    size_t small_bytes = 0;
    cudaEvent_t e_h2d = nullptr, e_stft = nullptr, e_kernel = nullptr, e_done = nullptr;
    cudaEvent_t t_h2d0 = nullptr, t_d2h0 = nullptr;   // SPX_RING_TRACE=1 only: start of the H2D / of the rows' D2H
    long long seq = -1, n_frames = 0, first_frame = 0, h2d_bytes = 0, d2h_bytes = 0;
    bool has_features = false;
    int state = 0;                   // 0 free, 1 acquired (being filled), 2 committed (in flight / ready)
};

}  // namespace spx

namespace spx {
// the (nfft - hop)-sample tail of a slot, copied to the head of the next slot's device buffer (sample sizes are multiples of 4 bytes)
__global__ void __launch_bounds__(256) ring_carry_kernel(unsigned int* __restrict__ dst, const unsigned int* __restrict__ src, unsigned n_words) {
    const unsigned i = blockIdx.x * 256u + threadIdx.x;
    if (i < n_words) dst[i] = src[i];
}
}  // namespace spx

struct spx_ring {
    spx_plan* plan = nullptr;
    spx_ring_config cfg{};
    std::vector<spx::RingSlot> slots;
    size_t elt = 8;
    long long frames_max = 0;
    int head = 0;                    // next slot to acquire
    int tail = 0;                    // oldest committed slot not yet released
    int in_flight = 0;
    long long seq = 0;
    long long carry = 0;             // samples already on the device that the next frames start in
    long long frames_total = 0, samples_total = 0, h2d_total = 0, d2h_total = 0;
    bool trace = false;              // SPX_RING_TRACE=1: timed events, one timeline line per released slot on stderr
    cudaEvent_t e_ref = nullptr;
    std::mutex mu;
};

using namespace spx;

static void ring_free(spx_ring* r) {
    for (RingSlot& s : r->slots) {
        if (s.h_in) cudaFreeHost(s.h_in);
        if (s.d_in) cudaFree(s.d_in);
        if (s.d_wf) cudaFree(s.d_wf);
        if (s.h_wf) cudaFreeHost(s.h_wf);
        if (s.d_db) cudaFree(s.d_db);
        if (s.h_db) cudaFreeHost(s.h_db);
        if (s.d_small) cudaFree(s.d_small);
        if (s.h_small) cudaFreeHost(s.h_small);
        if (s.e_h2d) cudaEventDestroy(s.e_h2d);
        if (s.e_stft) cudaEventDestroy(s.e_stft);
        if (s.t_h2d0) cudaEventDestroy(s.t_h2d0);
        if (s.t_d2h0) cudaEventDestroy(s.t_d2h0);
        if (s.e_kernel) cudaEventDestroy(s.e_kernel);
        if (s.e_done) cudaEventDestroy(s.e_done);
    }
    if (r->e_ref) cudaEventDestroy(r->e_ref);
    delete r;
}

extern "C" int spx_ring_create(spx_ring** out, spx_plan* plan, const spx_ring_config* cfg) {
    if (!out || !plan || !cfg) return spx_set_error(SPX_E_INVALID, "NULL argument");
    *out = nullptr;
    if (cfg->struct_size != sizeof(spx_ring_config)) return spx_set_error(SPX_E_INVALID, "spx_ring_config.struct_size mismatch");
    if (cfg->n_slots < 2 || cfg->n_slots > 64) return spx_set_error(SPX_E_INVALID, "n_slots must be in [2, 64]");
    if (cfg->slot_samples < plan->cfg.nfft) return spx_set_error(SPX_E_INVALID, "slot_samples must be >= nfft");
    if (cfg->want_wf_rows && !(cfg->vmax > cfg->vmin)) return spx_set_error(SPX_E_INVALID, "wf rows need vmax > vmin");
    if (cfg->want_features && (!cfg->want_welch || !(cfg->sample_rate > 0)))
        return spx_set_error(SPX_E_INVALID, "want_features needs want_welch and a positive sample_rate");
    SPX_CUDA(cudaSetDevice(plan->cfg.device));
    spx_ring* r = new (std::nothrow) spx_ring();
    if (!r) return spx_set_error(SPX_E_NOMEM, "out of host memory");
    r->plan = plan;
    r->cfg = *cfg;
    r->elt = plan->cfg.in_fmt == SPX_FMT_CI16 ? 4 : 8;
    const size_t N = (size_t)plan->cfg.nfft;
    r->frames_max = (cfg->slot_samples + (long long)N) / plan->cfg.hop + 1;
    r->slots.resize((size_t)cfg->n_slots);
    cudaError_t e = cudaSuccess;
    const char* tr = getenv("SPX_RING_TRACE");
    r->trace = tr != nullptr && tr[0] == '1';
    if (r->trace) {
        cudaEventCreate(&r->e_ref);
        cudaEventRecord(r->e_ref, plan->s_h2d);
    }
    for (RingSlot& s : r->slots) {
        const size_t rows = (size_t)r->frames_max * N;
        if ((e = cudaHostAlloc(&s.h_in, (size_t)cfg->slot_samples * r->elt, cudaHostAllocPortable)) != cudaSuccess) break;
        if ((e = cudaMalloc((void**)&s.d_in, (N + (size_t)cfg->slot_samples) * r->elt)) != cudaSuccess) break;
        if (cfg->want_wf_rows) {
            if ((e = cudaMalloc((void**)&s.d_wf, rows)) != cudaSuccess) break;
            if ((e = cudaHostAlloc((void**)&s.h_wf, rows, cudaHostAllocPortable)) != cudaSuccess) break;
        }
        if (cfg->want_db_rows) {
            if ((e = cudaMalloc((void**)&s.d_db, rows * sizeof(float))) != cudaSuccess) break;
            if ((e = cudaHostAlloc((void**)&s.h_db, rows * sizeof(float), cudaHostAllocPortable)) != cudaSuccess) break;
        }
        {
            size_t off = 0, o_welch = 0, o_pdb = 0, o_max = 0, o_feat = 0;
            if (cfg->want_welch) { o_welch = off; off += N * sizeof(double); }
            if (cfg->want_features) { o_pdb = off; off += N * sizeof(double); }
            if (cfg->want_maxhold) { o_max = off; off += N * sizeof(float); }
            off = (off + 7) & ~(size_t)7;
            if (cfg->want_features) { o_feat = off; off += sizeof(spx_features); }
            s.small_bytes = off;
            if (off) {
                if ((e = cudaMalloc((void**)&s.d_small, off)) != cudaSuccess) break;
                if ((e = cudaHostAlloc((void**)&s.h_small, off, cudaHostAllocPortable)) != cudaSuccess) break;
                memset(s.h_small, 0, off);
                if (cfg->want_welch) { s.d_welch = (double*)(s.d_small + o_welch); s.h_welch = (double*)(s.h_small + o_welch); }
                if (cfg->want_maxhold) { s.d_max = (float*)(s.d_small + o_max); s.h_max = (float*)(s.h_small + o_max); }
                if (cfg->want_features) {
                    s.d_pdb = (double*)(s.d_small + o_pdb); s.h_pdb = (double*)(s.h_small + o_pdb);
                    s.d_feat = (spx_features*)(s.d_small + o_feat); s.h_feat = (spx_features*)(s.h_small + o_feat);
                }
            }
        }
        const unsigned evf = r->trace ? cudaEventDefault : cudaEventDisableTiming;
        if ((e = cudaEventCreateWithFlags(&s.e_h2d, evf)) != cudaSuccess) break;
        if ((e = cudaEventCreateWithFlags(&s.e_stft, evf)) != cudaSuccess) break;
        if ((e = cudaEventCreateWithFlags(&s.e_kernel, evf)) != cudaSuccess) break;
        if ((e = cudaEventCreateWithFlags(&s.e_done, evf)) != cudaSuccess) break;
        if (r->trace) {
            if ((e = cudaEventCreate(&s.t_h2d0)) != cudaSuccess) break;
            if ((e = cudaEventCreate(&s.t_d2h0)) != cudaSuccess) break;
        }
    }
    if (e != cudaSuccess) {
        ring_free(r);
        return spx_set_error(SPX_E_NOMEM, "ring allocation failed: %s", cudaGetErrorString(e));
    }
    *out = r;
    return SPX_OK;
}

extern "C" int spx_ring_destroy(spx_ring* r) {
    if (!r) return SPX_OK;
    cudaSetDevice(r->plan->cfg.device);
    cudaStreamSynchronize(r->plan->s_h2d);
    cudaStreamSynchronize(r->plan->s_h2d_alt);
    cudaStreamSynchronize(r->plan->s_compute);
    cudaStreamSynchronize(r->plan->s_d2h);
    ring_free(r);
    return SPX_OK;
}

extern "C" int spx_ring_acquire(spx_ring* r, void** host_slot, int64_t* capacity_samples) {
    if (!r || !host_slot) return spx_set_error(SPX_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(r->mu);
    RingSlot& s = r->slots[(size_t)r->head];
    if (s.state != 0) return spx_set_error(SPX_E_BUSY, "ring full: collect/release the oldest slot first");
    s.state = 1;
    *host_slot = s.h_in;
    if (capacity_samples) *capacity_samples = r->cfg.slot_samples;
    return SPX_OK;
}

extern "C" int spx_ring_commit(spx_ring* r, int64_t n_samples) {
    if (!r) return spx_set_error(SPX_E_INVALID, "ring is NULL");
    std::lock_guard<std::mutex> g(r->mu);
    RingSlot& s = r->slots[(size_t)r->head];
    if (s.state != 1) return spx_set_error(SPX_E_INVALID, "commit without acquire");
    if (n_samples < 0 || n_samples > r->cfg.slot_samples) return spx_set_error(SPX_E_INVALID, "n_samples out of range");
    spx_plan* pl = r->plan;
    std::lock_guard<std::mutex> gp(pl->mu);
    SPX_CUDA(cudaSetDevice(pl->cfg.device));
    const int N = pl->cfg.nfft, hop = pl->cfg.hop;
    const size_t elt = r->elt;
    const long long carry = r->carry;
    NvtxRange r_commit("spx ring commit: H2D -> STFT -> D2H");
    // H2D of the new samples behind the carried tail
    cudaStream_t s_up = (r->seq & 1) ? pl->s_h2d_alt : pl->s_h2d;   // consecutive slots upload on alternating streams (spx_plan.h)
    if (r->trace) SPX_CUDA(cudaEventRecord(s.t_h2d0, s_up));
    if (n_samples) SPX_CUDA(cudaMemcpyAsync(s.d_in + (size_t)carry * elt, s.h_in, (size_t)n_samples * elt, cudaMemcpyHostToDevice, s_up));
    SPX_CUDA(cudaEventRecord(s.e_h2d, s_up));
    SPX_CUDA(cudaStreamWaitEvent(pl->s_compute, s.e_h2d, 0));
    const long long avail = carry + n_samples;
    const long long F = spx_frame_count(avail, N, hop);
    if (s.d_welch) SPX_CUDA(cudaMemsetAsync(s.d_welch, 0, (size_t)N * sizeof(double), pl->s_compute));
    if (s.d_max) SPX_CUDA(cudaMemsetAsync(s.d_max, 0, (size_t)N * sizeof(float), pl->s_compute));
    // a one-shot call on the same plan may still be using its scratch on a caller stream, and one enqueued after this
    // commit must wait for the slot's kernels
    const bool scratch = plan_has_scratch(pl);
    if (scratch) SPX_TRY(scratch_wait(pl, pl->s_compute));
    SPX_TRY(stft_launch_device(pl, s.d_in, 1, 0, F, StftOut{s.d_db, s.d_wf, nullptr, s.d_welch, s.d_max, r->cfg.vmin, r->cfg.vmax},
                               pl->s_compute));
    SPX_CUDA(cudaEventRecord(s.e_stft, pl->s_compute));   // the rows are complete here: their copy does not wait for the measurements
    // classifier measurements of this slot's Welch block, right behind the STFT kernel on the same stream
    const bool feats = s.d_feat != nullptr && F > 0;
    if (feats) {
        const double inv = 1.0 / ((double)F * r->cfg.sample_rate * pl->sum_w2);
        SPX_TRY(welch_finalize_launch(s.d_welch, N, inv, nullptr, s.d_pdb, pl->s_compute));
        SPX_TRY(spx_classify_features_dev(pl->cfg.device, s.d_pdb, 1, N, 1, N, s.d_feat, nullptr, 0, nullptr, pl->s_compute));
    }
    if (scratch) SPX_TRY(scratch_record(pl, pl->s_compute));
    // carry the unconsumed tail into the head of the next slot's device buffer
    const long long consumed = F * hop;
    const long long new_carry = avail - consumed;
    RingSlot& nx = r->slots[(size_t)((r->head + 1) % r->cfg.n_slots)];
    if (new_carry > 0) {
        // a kernel, not cudaMemcpyAsync: a device-to-device copy would go to a copy engine and sit between the H2D / D2H transfers
        const unsigned n_words = (unsigned)((size_t)new_carry * elt / 4);
        ring_carry_kernel<<<(n_words + 255) / 256, 256, 0, pl->s_compute>>>(reinterpret_cast<unsigned int*>(nx.d_in),
                                                                             reinterpret_cast<const unsigned int*>(s.d_in + (size_t)consumed * elt), n_words);
        SPX_CUDA(cudaGetLastError());
    }
    SPX_CUDA(cudaEventRecord(s.e_kernel, pl->s_compute));
    // drain the slot's results: the rows as soon as the STFT kernel is done, the small block (one copy) behind the measurements
    long long d2h = 0;
    SPX_CUDA(cudaStreamWaitEvent(pl->s_d2h, s.e_stft, 0));
    if (r->trace) SPX_CUDA(cudaEventRecord(s.t_d2h0, pl->s_d2h));
    if (s.d_wf && F) { SPX_CUDA(cudaMemcpyAsync(s.h_wf, s.d_wf, (size_t)F * N, cudaMemcpyDeviceToHost, pl->s_d2h)); d2h += F * N; }
    if (s.d_db && F) { SPX_CUDA(cudaMemcpyAsync(s.h_db, s.d_db, (size_t)F * N * sizeof(float), cudaMemcpyDeviceToHost, pl->s_d2h)); d2h += F * N * 4; }
    SPX_CUDA(cudaStreamWaitEvent(pl->s_d2h, s.e_kernel, 0));
    if (s.small_bytes) {
        SPX_CUDA(cudaMemcpyAsync(s.h_small, s.d_small, s.small_bytes, cudaMemcpyDeviceToHost, pl->s_d2h));
        d2h += (long long)s.small_bytes;
    }
    s.has_features = feats;
    SPX_CUDA(cudaEventRecord(s.e_done, pl->s_d2h));
    s.seq = r->seq++;
    s.n_frames = F;
    s.first_frame = r->frames_total;
    s.h2d_bytes = n_samples * (long long)elt;
    s.d2h_bytes = d2h;
    s.state = 2;
    r->carry = new_carry;
    r->frames_total += F;
    r->samples_total += n_samples;
    r->h2d_total += s.h2d_bytes;
    r->d2h_total += d2h;
    r->head = (r->head + 1) % r->cfg.n_slots;
    r->in_flight++;
    return SPX_OK;
}

extern "C" int spx_ring_collect(spx_ring* r, spx_ring_result* out) {
    if (!r || !out) return spx_set_error(SPX_E_INVALID, "NULL argument");
    RingSlot* s;
    {
        std::lock_guard<std::mutex> g(r->mu);
        if (r->in_flight == 0) return spx_set_error(SPX_E_BUSY, "nothing committed");
        s = &r->slots[(size_t)r->tail];
    }
    SPX_CUDA(cudaEventSynchronize(s->e_done));   // outside the lock: the producer may keep committing
    memset(out, 0, sizeof(*out));
    out->struct_size = sizeof(*out);
    out->seq = s->seq;
    out->n_frames = s->n_frames;
    out->first_frame = s->first_frame;
    out->wf_rows = s->h_wf;
    out->db_rows = s->h_db;
    out->welch_acc = s->h_welch;
    out->maxhold = s->h_max;
    out->h2d_bytes = s->h2d_bytes;
    out->d2h_bytes = s->d2h_bytes;
    out->pxx_db = s->has_features ? s->h_pdb : nullptr;
    out->features = s->has_features ? s->h_feat : nullptr;
    return SPX_OK;
}

extern "C" int spx_ring_release(spx_ring* r) {
    if (!r) return spx_set_error(SPX_E_INVALID, "ring is NULL");
    std::lock_guard<std::mutex> g(r->mu);
    if (r->in_flight == 0) return spx_set_error(SPX_E_BUSY, "nothing to release");
    RingSlot& s = r->slots[(size_t)r->tail];
    SPX_CUDA(cudaEventSynchronize(s.e_done));
    if (r->trace) {
        float t[6] = {0, 0, 0, 0, 0, 0};
        cudaEvent_t ev[6] = {s.t_h2d0, s.e_h2d, s.e_stft, s.e_kernel, s.t_d2h0, s.e_done};
        for (int i = 0; i < 6; ++i) cudaEventElapsedTime(&t[i], r->e_ref, ev[i]);
        fprintf(stderr, "spx_ring_trace seq %lld us: h2d %.0f..%.0f stft_done %.0f meas_done %.0f d2h %.0f..%.0f\n", s.seq, t[0] * 1e3,
                t[1] * 1e3, t[2] * 1e3, t[3] * 1e3, t[4] * 1e3, t[5] * 1e3);
    }
    s.state = 0;
    r->tail = (r->tail + 1) % r->cfg.n_slots;
    r->in_flight--;
    return SPX_OK;
}

extern "C" int spx_ring_stats(spx_ring* r, spx_ring_stats_t* out) {
    if (!r || !out) return spx_set_error(SPX_E_INVALID, "NULL argument");
    std::lock_guard<std::mutex> g(r->mu);
    out->struct_size = sizeof(*out);
    out->h2d_bytes = r->h2d_total;
    out->d2h_bytes = r->d2h_total;
    out->samples = r->samples_total;
    out->frames = r->frames_total;
    out->in_flight = r->in_flight;
    out->reserved = 0;
    return SPX_OK;
}
