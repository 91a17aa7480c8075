// spx_fir.h -- the handle state, set-up, argument checks and host-memory pipeline that the FIR handles (DDC, channelizer)
// share.  Each handle derives from FirHandle and adds its own config, launch geometry and kernel launch.
#pragma once
#include <cuda_runtime.h>

#include <mutex>
#include <vector>

#include "spx_internal.h"
#include "spx_plan.h"

namespace spx {

// cudaMalloc + upload of a host table: SPX_E_NOMEM when the allocation fails
template <class T>
int upload(T** dst, const std::vector<T>& src) {
    const cudaError_t e = cudaMalloc(dst, src.size() * sizeof(T));
    if (e != cudaSuccess) return spx_set_error(SPX_E_NOMEM, "%s", cudaGetErrorString(e));
    SPX_CUDA(cudaMemcpy(*dst, src.data(), src.size() * sizeof(T), cudaMemcpyHostToDevice));
    return SPX_OK;
}

// check_device, then the limits a FIR handle's launch planning needs
inline int fir_device(int device, int* max_smem, int* sm_count) {
    SPX_TRY(check_device(device));
    SPX_CUDA(cudaDeviceGetAttribute(max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    SPX_CUDA(cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, device));
    return SPX_OK;
}

struct FirHandle {
    int device = 0, in_fmt = 0, n_taps = 0, decim = 0;
    float in_scale = 1.0f;
    int sm_count = 0, max_smem = 0;   // max_smem: the device's opt-in dynamic shared memory per block
    const void* kern = nullptr;       // the one kernel this handle launches
    float* d_taps = nullptr;          // reversed, float32
    cudaStream_t s_compute = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    std::vector<cudaEvent_t> events;  // of the host-memory pipeline, grown on demand
    size_t piece_bytes = 16u << 20;   // H2D piece of the host path (SPX_H2D_PIECE_BYTES)
    DevBuf st_in, st_out;             // staging of the host path: two input pieces, the handle's outputs
    std::mutex mu;

    size_t elt() const { return in_fmt == SPX_FMT_CI16 ? 4 : 8; }
    long long out_count(long long L) const { return L < n_taps ? 0 : (L - n_taps) / decim + 1; }

    // After the handle's own config checks and launch planning (fir_device gave max_smem and sm_count): keeps the
    // config's common fields, uploads the reversed taps rounded once to float32, reads SPX_H2D_PIECE_BYTES, raises
    // `kernel`'s dynamic shared-memory limit to max_smem and creates the three streams.
    template <class Cfg>
    int setup(const Cfg& cfg, const void* kernel, int max_smem_optin, int sms) {
        device = cfg.device;
        in_fmt = cfg.in_fmt;
        in_scale = cfg.in_scale != 0.0f ? cfg.in_scale : 1.0f;
        n_taps = cfg.n_taps;
        decim = cfg.decim;
        sm_count = sms;
        max_smem = max_smem_optin;
        kern = kernel;
        std::vector<float> g((size_t)n_taps);
        for (int j = 0; j < n_taps; ++j) g[(size_t)j] = (float)cfg.taps[n_taps - 1 - j];
        SPX_TRY(upload(&d_taps, g));
        piece_bytes = env_bytes("SPX_H2D_PIECE_BYTES", piece_bytes, 65536);
        SPX_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem));
        for (cudaStream_t* s : {&s_compute, &s_h2d, &s_d2h}) SPX_CUDA(cudaStreamCreateWithFlags(s, cudaStreamNonBlocking));
        return SPX_OK;
    }

    // Waits for and destroys the streams, then frees the events, the taps and the staging.
    void release() {
        cudaSetDevice(device);
        for (cudaStream_t s : {s_compute, s_h2d, s_d2h})
            if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); }
        for (cudaEvent_t e : events) cudaEventDestroy(e);
        if (d_taps) cudaFree(d_taps);
        st_in.release();
        st_out.release();
    }

    int sync() {
        std::lock_guard<std::mutex> g(mu);
        SPX_CUDA(cudaSetDevice(device));
        SPX_CUDA(cudaStreamSynchronize(s_h2d));
        SPX_CUDA(cudaStreamSynchronize(s_compute));
        SPX_CUDA(cudaStreamSynchronize(s_d2h));
        return SPX_OK;
    }

    // The checks of an exec call, in this order: mem, n_samples, first_sample; then *M = the output count (also to n_out)
    // and zero byte counters; nothing more when *M == 0; then out and in non-NULL, in 4-byte and out out_align-byte
    // aligned.  On SPX_OK with *M > 0 the handle is locked in `lock` and its device is current.
    int exec_begin(int32_t mem, const void* in, int64_t n_samples, int64_t first_sample, const void* out,
                   uintptr_t out_align, long long* M, int64_t* n_out, int64_t* h2d_bytes_out, int64_t* d2h_bytes_out,
                   std::unique_lock<std::mutex>* lock) {
        if (mem != SPX_MEM_HOST && mem != SPX_MEM_DEVICE) return spx_set_error(SPX_E_INVALID, "unknown mem %d", mem);
        if (n_samples < 0) return spx_set_error(SPX_E_INVALID, "n_samples < 0");
        if (first_sample < 0) return spx_set_error(SPX_E_INVALID, "first_sample < 0");
        *M = out_count(n_samples);
        if (n_out) *n_out = *M;
        if (h2d_bytes_out) *h2d_bytes_out = 0;
        if (d2h_bytes_out) *d2h_bytes_out = 0;
        if (*M == 0) return SPX_OK;
        if (!out) return spx_set_error(SPX_E_INVALID, "out is NULL");
        if (!in) return spx_set_error(SPX_E_INVALID, "in is NULL");
        if (((uintptr_t)in & 3u) || ((uintptr_t)out & (out_align - 1)))
            return spx_set_error(SPX_E_INVALID, "in must be 4-byte and out %d-byte aligned", (int)out_align);
        *lock = std::unique_lock<std::mutex>(mu);
        SPX_CUDA(cudaSetDevice(device));
        return SPX_OK;
    }

    // Outputs per piece of the host path over M outputs: about piece_bytes of input each.
    long long piece_outputs(long long M) const {
        long long per = ((long long)(piece_bytes / elt()) - n_taps) / decim + 1;
        if (per < 1) per = 1;
        if (per > M) per = M;
        return per;
    }

    // M outputs of host input `in` in pieces of `per` outputs: piece k covers outputs [m0, m0 + nm) and input samples
    // [m0 D, m0 D + (nm - 1) D + T), i.e. consecutive pieces overlap by the T - D halo.  Each piece is uploaded on s_h2d
    // into one of two alternating buffers (the upload of piece k + 1 overlaps the kernel of piece k), then
    //   launch(d_in, n, a, m0, nm, b, s_compute)   enqueues the kernel on samples [a, a + n) of the call, in buffer b's turn;
    //   drain(m0, nm, b, s_d2h, &bytes)            enqueues the copy of the piece's outputs to the host.
    // With out_buffers_alternate, a launch in buffer b's turn also waits for the drain of the piece before it in that turn,
    // so the handle may stage its outputs in two alternating buffers; without it the kernels never wait for a copy to the
    // host.  Returns when every copy has landed, with the bytes copied each way in *h2d_out and *d2h_out (if non-NULL).
    template <class Launch, class Drain>
    int host_pieces(const void* in, long long M, long long per, bool out_buffers_alternate, Launch launch, Drain drain,
                    int64_t* h2d_out, int64_t* d2h_out) {
        const int T = n_taps, D = decim;
        const size_t elt = this->elt();
        const long long span = (per - 1) * D + T;   // input samples of a full piece
        SPX_TRY(st_in.reserve(2 * (size_t)span * elt));
        char* d_in[2] = {(char*)st_in.ptr, (char*)st_in.ptr + (size_t)span * elt};
        long long h2d = 0, d2h = 0;
        size_t ev = 0;
        cudaEvent_t e_read[2] = {nullptr, nullptr}, e_drained[2] = {nullptr, nullptr};
        for (long long m0 = 0, k = 0; m0 < M; m0 += per, ++k) {
            const long long nm = M - m0 < per ? M - m0 : per;
            const long long a = m0 * D, n = (nm - 1) * D + T;
            const int b = (int)(k & 1);
            cudaEvent_t e_in, e_k, e_d;
            SPX_TRY(event_at(events, ev++, &e_in));
            SPX_TRY(event_at(events, ev++, &e_k));
            SPX_TRY(event_at(events, ev++, &e_d));
            if (e_read[b]) SPX_CUDA(cudaStreamWaitEvent(s_h2d, e_read[b], 0));   // the kernel that last read this buffer
            SPX_CUDA(cudaMemcpyAsync(d_in[b], (const char*)in + (size_t)a * elt, (size_t)n * elt, cudaMemcpyHostToDevice,
                                     s_h2d));
            h2d += n * (long long)elt;
            SPX_CUDA(cudaEventRecord(e_in, s_h2d));
            SPX_CUDA(cudaStreamWaitEvent(s_compute, e_in, 0));
            if (out_buffers_alternate && e_drained[b]) SPX_CUDA(cudaStreamWaitEvent(s_compute, e_drained[b], 0));
            SPX_TRY(launch((const void*)d_in[b], n, a, m0, nm, b, s_compute));
            SPX_CUDA(cudaEventRecord(e_k, s_compute));
            e_read[b] = e_k;
            SPX_CUDA(cudaStreamWaitEvent(s_d2h, e_k, 0));
            long long bytes = 0;
            SPX_TRY(drain(m0, nm, b, s_d2h, &bytes));
            d2h += bytes;
            SPX_CUDA(cudaEventRecord(e_d, s_d2h));
            e_drained[b] = e_d;
        }
        SPX_CUDA(cudaStreamSynchronize(s_h2d));
        SPX_CUDA(cudaStreamSynchronize(s_compute));
        SPX_CUDA(cudaStreamSynchronize(s_d2h));
        if (h2d_out) *h2d_out = h2d;
        if (d2h_out) *d2h_out = d2h;
        return SPX_OK;
    }
};

}  // namespace spx
