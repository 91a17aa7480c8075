// spx_pieces.h -- the host-memory pipeline of the FIR handles (DDC, channelizer): input pieces cut at output boundaries.
#pragma once
#include <cuda_runtime.h>

#include <vector>

#include "spx_internal.h"
#include "spx_plan.h"

namespace spx {

// Streams and staging of a handle's host-memory calls.
struct HostPieces {
    cudaStream_t s_h2d, s_compute, s_d2h;
    std::vector<cudaEvent_t>* events;   // grown on demand, owned by the handle
    DevBuf* st_in;                      // two input pieces
    size_t piece_bytes;                 // SPX_H2D_PIECE_BYTES
    bool out_buffers_alternate;         // the launches write two alternating output buffers (see host_pieces)
};

inline int piece_event(std::vector<cudaEvent_t>& ev, size_t i, cudaEvent_t* out) {
    while (ev.size() <= i) {
        cudaEvent_t e;
        SPX_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        ev.push_back(e);
    }
    *out = ev[i];
    return SPX_OK;
}

// Outputs per piece of a FIR with T taps and decimation D over M outputs: about piece_bytes of input each.
inline long long piece_outputs(size_t piece_bytes, size_t elt, int T, int D, long long M) {
    long long per = ((long long)(piece_bytes / elt) - T) / D + 1;
    if (per < 1) per = 1;
    if (per > M) per = M;
    return per;
}

// M outputs of host input `in` (elt bytes a sample) in pieces of `per` outputs: piece k covers outputs [m0, m0 + nm) and
// input samples [m0 D, m0 D + (nm - 1) D + T), i.e. consecutive pieces overlap by the T - D halo.  Each piece is uploaded
// on s_h2d into one of two alternating buffers (the upload of piece k + 1 overlaps the kernel of piece k), then
//   launch(d_in, n, a, m0, nm, b, s_compute)   enqueues the kernel on samples [a, a + n) of the call, in buffer b's turn;
//   drain(m0, nm, b, s_d2h, &bytes)            enqueues the copy of the piece's outputs to the host.
// With out_buffers_alternate, a launch in buffer b's turn also waits for the drain of the piece before it in that turn, so
// the handle may stage its outputs in two alternating buffers; without it the kernels never wait for a copy to the host.
// Returns when every copy has landed.
template <class Launch, class Drain>
int host_pieces(const HostPieces& hp, const void* in, size_t elt, int T, int D, long long M, long long per,
                Launch launch, Drain drain, int64_t* h2d_out, int64_t* d2h_out) {
    const long long span = (per - 1) * D + T;   // input samples of a full piece
    SPX_TRY(hp.st_in->reserve(2 * (size_t)span * elt));
    char* d_in[2] = {(char*)hp.st_in->ptr, (char*)hp.st_in->ptr + (size_t)span * elt};
    long long h2d = 0, d2h = 0;
    size_t ev = 0;
    cudaEvent_t e_read[2] = {nullptr, nullptr}, e_drained[2] = {nullptr, nullptr};
    for (long long m0 = 0, k = 0; m0 < M; m0 += per, ++k) {
        const long long nm = M - m0 < per ? M - m0 : per;
        const long long a = m0 * D, n = (nm - 1) * D + T;
        const int b = (int)(k & 1);
        cudaEvent_t e_in, e_k, e_d;
        SPX_TRY(piece_event(*hp.events, ev++, &e_in));
        SPX_TRY(piece_event(*hp.events, ev++, &e_k));
        SPX_TRY(piece_event(*hp.events, ev++, &e_d));
        if (e_read[b]) SPX_CUDA(cudaStreamWaitEvent(hp.s_h2d, e_read[b], 0));   // the kernel that last read this buffer
        SPX_CUDA(cudaMemcpyAsync(d_in[b], (const char*)in + (size_t)a * elt, (size_t)n * elt, cudaMemcpyHostToDevice,
                                 hp.s_h2d));
        h2d += n * (long long)elt;
        SPX_CUDA(cudaEventRecord(e_in, hp.s_h2d));
        SPX_CUDA(cudaStreamWaitEvent(hp.s_compute, e_in, 0));
        if (hp.out_buffers_alternate && e_drained[b]) SPX_CUDA(cudaStreamWaitEvent(hp.s_compute, e_drained[b], 0));
        SPX_TRY(launch((const void*)d_in[b], n, a, m0, nm, b, hp.s_compute));
        SPX_CUDA(cudaEventRecord(e_k, hp.s_compute));
        e_read[b] = e_k;
        SPX_CUDA(cudaStreamWaitEvent(hp.s_d2h, e_k, 0));
        long long bytes = 0;
        SPX_TRY(drain(m0, nm, b, hp.s_d2h, &bytes));
        d2h += bytes;
        SPX_CUDA(cudaEventRecord(e_d, hp.s_d2h));
        e_drained[b] = e_d;
    }
    SPX_CUDA(cudaStreamSynchronize(hp.s_h2d));
    SPX_CUDA(cudaStreamSynchronize(hp.s_compute));
    SPX_CUDA(cudaStreamSynchronize(hp.s_d2h));
    *h2d_out = h2d;
    *d2h_out = d2h;
    return SPX_OK;
}

}  // namespace spx
