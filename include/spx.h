/* spx.h -- C ABI of libspx: the B200-native spectral hot path of sdr-iq-visualizer.
 *
 * The reference (JaredWinkens/sdr-iq-visualizer) is pure Python and has no FFI of its own; its
 * boundary for this path is a set of Python call sites (SURVEY.md section 8(b)).  Each entry
 * point below names the reference lines it replaces.  The Python host layer
 * (sdr_iq_visualizer_b200/_native.py) binds exactly these symbols with ctypes; INTEGRATION.md shows
 * the stub a reference maintainer would add.
 *
 * Conventions
 *   - every function returns an int status: SPX_OK (0) or a negative SPX_E_* code; the message
 *     is available from spx_last_error() (thread-local).  No C++ exception crosses the boundary.
 *   - the caller owns every input and output buffer; a plan owns only scratch/staging memory.
 *   - `mem` says where the caller's buffers live: SPX_MEM_HOST (the library stages them through
 *     pinned memory with pipelined cudaMemcpyAsync) or SPX_MEM_DEVICE (pointers are used as is on
 *     `stream`; nothing is synchronised).
 *   - spectra are in fftshift order: index j <-> bin (j + N/2) mod N, freqs[j] = (j - N/2) fs/N + fc
 *     (reference app/sdr/streamer.py:119-120).
 *   - one plan may be used by one thread at a time (calls on the same plan are serialised by an
 *     internal mutex); different plans are independent.
 */
#ifndef SPX_H_
#define SPX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPX_ABI_VERSION 3

#if defined(__GNUC__)
#define SPX_API __attribute__((visibility("default")))
#else
#define SPX_API
#endif

/* status codes */
#define SPX_OK 0
#define SPX_E_INVALID (-1)     /* bad argument */
#define SPX_E_CUDA (-2)        /* CUDA runtime / launch failure */
#define SPX_E_NOMEM (-3)       /* allocation failed */
#define SPX_E_UNSUPPORTED (-4) /* e.g. nfft outside the supported range */
#define SPX_E_NODEVICE (-5)    /* no CUDA device: there is NO CPU fallback */
#define SPX_E_BUSY (-6)        /* ring full / nothing to collect */

/* enums */
#define SPX_WINDOW_RECT 0     /* streamer.py:119 (no window) */
#define SPX_WINDOW_HANN 1     /* np.hanning: mlab default behind process_sigmf_data.py:188 */
#define SPX_WINDOW_BLACKMAN 2 /* np.blackman */
#define SPX_FMT_CF32 0        /* complex64 (SigMF cf32_le; callbacks.py:307-310) */
#define SPX_FMT_CI16 1        /* interleaved int16 I,Q (Pluto iio buffer; SigMF ci16_le) */
#define SPX_MEM_HOST 0
#define SPX_MEM_DEVICE 1

SPX_API int spx_abi_version(void);
/* thread-local message of the last failing call on this thread ("" if none) */
SPX_API const char* spx_last_error(void);

SPX_API int spx_device_count(int* count);

typedef struct {
    uint32_t struct_size;
    int32_t sm_count;
    int32_t cc_major, cc_minor;
    int32_t l2_bytes;
    int32_t max_smem_optin;
    int64_t total_mem;
    char name[64];
} spx_device_info;
SPX_API int spx_get_device_info(int device, spx_device_info* out);

/* F = (n_samples - nfft) / hop + 1 (0 if n_samples < nfft): frame slicing of SURVEY.md A2
 * (one rx buffer = one frame at streamer.py:114-119; mlab framing behind process_sigmf_data.py:188) */
SPX_API int64_t spx_frame_count(int64_t n_samples, int32_t nfft, int32_t hop);

/* Measured FP32 peak of the device: an FFMA micro-kernel (8 independent chains per thread, every SM full), best of
 * 5 launches timed with CUDA events.  tflops_out = 2 * lane-FMAs / time.  bench.py reports the STFT kernel's FP32
 * pipe share against it (SURVEY.md 8(d): "measure P32 with an FMA micro-kernel in the same run"). */
SPX_API int spx_fp32_peak(int device, double* tflops_out);

/* ---------------------------------------------------------------- pinned host memory */
SPX_API int spx_host_alloc(void** out, size_t bytes);
/* write-combined pinned memory: for buffers the CPU only WRITES sequentially and the GPU reads over PCIe (ring slots,
 * staged input); CPU reads from it are slow.  Free with spx_host_free. */
SPX_API int spx_host_alloc_wc(void** out, size_t bytes);
SPX_API int spx_host_free(void* p);
SPX_API int spx_host_register(void* p, size_t bytes);
SPX_API int spx_host_unregister(void* p);

/* ---------------------------------------------------------------- device memory (for callers
 * that keep data resident, e.g. bench.py's device-timed leg and the multi-GPU sharder) */
SPX_API int spx_device_alloc(int device, void** out, size_t bytes);
SPX_API int spx_device_free(int device, void* p);
SPX_API int spx_memcpy_h2d(int device, void* dst, const void* src, size_t bytes);
SPX_API int spx_memcpy_d2h(int device, void* dst, const void* src, size_t bytes);
SPX_API int spx_memcpy_d2h_async(int device, void* dst_host, const void* src, size_t bytes, void* stream);
SPX_API int spx_memset(int device, void* dst, int value, size_t bytes);
SPX_API int spx_device_sync(int device);
/* device -> device copy on `stream`; either pointer may be a peer GPU's buffer mapped with spx_ipc_open (NVLink) */
SPX_API int spx_memcpy_d2d_async(int device, void* dst, const void* src, size_t bytes, void* stream);
SPX_API int spx_stream_sync(int device, void* stream);
/* side streams for callers that overlap SPX_MEM_DEVICE calls (e.g. the classifier measurements of Welch block k next to
 * the STFT of block k+1): everything enqueued on `waiter` after the call runs after what `signaller` holds now */
SPX_API int spx_stream_create(int device, void** stream_out);
SPX_API int spx_stream_destroy(int device, void* stream);
SPX_API int spx_stream_wait_stream(int device, void* waiter, void* signaller);

/* Measured copy ceiling of THIS box for the end-to-end path: h2d_bytes from `host_in` and d2h_bytes into `host_out`
 * (the caller's own pinned buffers) move concurrently on two streams in `piece_bytes` pieces, nothing else running;
 * seconds_out = wall time per repetition (mean of `iters` after one warm-up).  bench.py prints the end-to-end step
 * time against it (e2e.frac_of_copy_ceiling), per rank and with all ranks copying at once. */
SPX_API int spx_copy_ceiling(int device, const void* host_in, size_t h2d_bytes, void* host_out, size_t d2h_bytes,
                             size_t piece_bytes, int iters, double* seconds_out);

/* ---------------------------------------------------------------- peer memory (one process per GPU)
 * The multi-GPU configs reduce partial Welch sums / max-holds and collect waterfall rows on one rank
 * (SURVEY.md section 8(e)).  Instead of a separate collective, the owner exports its buffers and every rank's
 * STFT kernel writes / reduces straight into them over NVLink (spx_stft_args.peer_outputs).
 * spx_ipc_export: `dptr` must be the base of an allocation made by spx_device_alloc. */
#define SPX_IPC_HANDLE_BYTES 64
SPX_API int spx_ipc_export(int device, void* dptr, void* handle_out);
SPX_API int spx_ipc_open(int device, const void* handle, void** dptr_out);
SPX_API int spx_ipc_close(int device, void* dptr);

/* The collective step of a sharded capture (SURVEY.md 8(e); the reference is single-process, app/sdr/streamer.py:58),
 * for consumers that do not go through Python:
 *   spx_peer_reduce     adds this GPU's partial Welch sums (float64) / max-holds (float32, MAX) into the owner's
 *                       mapped buffers with system-scope atomics over NVLink (n = n_streams * nfft elements);
 *   spx_peer_push_rows  copy-engine push of a block of finished uint8 rows into the owner's mapped row buffer. */
SPX_API int spx_peer_reduce(int device, const double* welch_local, const float* maxhold_local, double* welch_owner,
                            float* maxhold_owner, int64_t n, void* stream);
SPX_API int spx_peer_push_rows(int device, void* rows_owner, const void* rows_local, size_t bytes, void* stream);

/* The same step over NCCL (libnccl.so.2 is loaded with dlopen at first use; SPX_NCCL_LIB overrides the path):
 *   spx_nccl_unique_id  rank 0 creates the 128-byte id and hands it to the other ranks out of band;
 *   spx_nccl_init       one communicator per process / GPU;
 *   spx_allreduce_welch in place: welch_acc SUM (float64[n]), maxhold MAX (float32[n]), *n_frames_inout SUM
 *                       (any of the three may be NULL); with n_frames_inout it waits for `stream`;
 *   spx_gather_rows     uint8 rows of every rank, in rank order, into rows_all on rank dst (bytes_per_rank[nranks]). */
typedef struct spx_comm spx_comm;
#define SPX_NCCL_ID_BYTES 128
SPX_API int spx_nccl_unique_id(void* id_out_128);
SPX_API int spx_nccl_init(spx_comm** out, int device, int rank, int nranks, const void* unique_id_128);
SPX_API int spx_nccl_destroy(spx_comm* comm);
SPX_API int spx_allreduce_welch(spx_comm* comm, double* welch_acc, float* maxhold, int64_t n, int64_t* n_frames_inout,
                                void* stream);
SPX_API int spx_gather_rows(spx_comm* comm, const void* rows_local, int64_t local_bytes, void* rows_all,
                            const int64_t* bytes_per_rank, int dst, void* stream);

/* The reference's per-buffer stream path in float64 (/root/reference/app/sdr/streamer.py:119-121): fftshift(fft(x)) and
 * 20*log10(|X| + eps), one rx buffer per call, power-of-two n in [2, 8192].  samples: complex128 (in_is_c128 = 1, what
 * pyadi-iio's rx() returns, :114) or complex64; power_db_out float64[n] / spec_out complex128[n] (both in fftshift
 * order) / wf_row uint8[n] (colormap index of the dB values, needs vmax > vmin): any subset.  With SPX_MEM_HOST the
 * call copies in and out and waits; with SPX_MEM_DEVICE it only enqueues on `stream`.  Agrees with numpy to ~1e-12 dB;
 * the batched STFT path (spx_stft_exec) computes in float32. */
SPX_API int spx_stream_frame_f64(int device, int mem, const void* samples, int in_is_c128, int n, double eps,
                                 double* power_db_out, double* spec_out, uint8_t* wf_row, double vmin, double vmax,
                                 void* stream);

/* ---------------------------------------------------------------- STFT plan */
typedef struct spx_plan spx_plan;

typedef struct {
    uint32_t struct_size; /* sizeof(spx_plan_config) */
    int32_t device;
    int32_t nfft;     /* power of two in [16, 1048576] (shared-memory / four-step kernels), or any length in
                       * [1, 524288] (Bluestein over the power-of-two kernels: the reference's np.fft.fft takes any
                       * rx_buffer_size, streamer.py:8-10,119) */
    int32_t hop;      /* 1 .. nfft (nfft = no overlap, nfft/4 = 75 % overlap) */
    int32_t window;   /* SPX_WINDOW_* */
    int32_t in_fmt;   /* SPX_FMT_* */
    float in_scale;   /* multiplies every sample: 1.0 stream path, 2^-15 SigMF ci16_le */
    float db_eps;     /* dB rows are 20*log10(|X| + db_eps); reference 1e-12 (streamer.py:121) */
    int32_t variant;  /* kernel selection; spx_plan_create rejects any other value with SPX_E_INVALID.  The non-zero
                       * values force a path the default also takes for some inputs, as a reference to test against;
                       * for lengths they do not concern they behave like 0.
                       *   0: the default (fastest measured kernel per shape)
                       *   1: N = 65536: the two-kernel four-step path instead of the single-kernel one
                       *  12: N = 1024 / 2048 / 4096: K1, the kernel the default uses for frames that are not 128-byte
                       *      aligned, for every input
                       *  22: N = 1024 / 2048 / 4096, aligned frames: the generic K1v2 kernel, without strip staging,
                       *      L2 prefetch or the kernels specialised to one set of row outputs */
    int32_t reserved;
} spx_plan_config;

SPX_API int spx_plan_create(spx_plan** out, const spx_plan_config* cfg);
SPX_API int spx_plan_destroy(spx_plan* plan);
/* wait for everything the plan has enqueued on its own streams */
SPX_API int spx_plan_sync(spx_plan* plan);

typedef struct {
    uint32_t struct_size; /* sizeof(spx_stft_args) */
    int32_t mem;          /* SPX_MEM_HOST or SPX_MEM_DEVICE, applies to every pointer below */
    const void* in;       /* n_streams streams of n_samples samples, stream s starts at s*stream_stride */
    int64_t n_samples;    /* per stream */
    int64_t stream_stride;/* in samples; ignored when n_streams == 1 */
    int32_t n_streams;    /* >= 1 */
    int32_t accumulate;   /* 0: welch_acc/maxhold are overwritten; 1: accumulated into (+=, max=) */
    /* outputs, each optional (NULL = not wanted); F = spx_frame_count(n_samples, nfft, hop) */
    float* db_rows;       /* [n_streams*F][nfft]  20*log10(|X|+eps), fftshift order (streamer.py:121) */
    uint8_t* wf_rows;     /* [n_streams*F][nfft]  clip(floor((db-vmin)*256/(vmax-vmin)),0,255) (A7) */
    float* spec_rows;     /* [n_streams*F][nfft][2] complex spectrum, fftshift order (streamer.py:119) */
    double* welch_acc;    /* [n_streams][nfft]    sum over frames of |X|^2 (A8; mlab.psd numerator) */
    float* maxhold;       /* [n_streams][nfft]    max over frames of |X|^2 (A8); NaN powers are skipped (fmax) */
    float vmin, vmax;     /* waterfall colour range in dB */
    void* stream;         /* cudaStream_t for SPX_MEM_DEVICE (NULL = the plan's compute stream) */
    int64_t n_frames_out; /* out: F */
    int64_t h2d_bytes_out;/* out: bytes copied host->device by this call (SPX_MEM_HOST) */
    int64_t d2h_bytes_out;/* out: bytes copied device->host by this call */
    int32_t peer_outputs; /* SPX_MEM_DEVICE only, bit mask.  bit 0: welch_acc / maxhold are shared with other GPUs (this
                           * GPU's or a peer's memory mapped with spx_ipc_open): partials are reduced locally and added
                           * with system-scope atomics, so several GPUs reduce into one buffer over NVLink.  bit 1:
                           * wf_rows lives on a peer GPU: rows are staged in frame pieces and pushed by the copy engine
                           * while the next piece is transformed */
    int32_t reserved;
} spx_stft_args;

/* windowed STFT -> PSD -> waterfall; replaces streamer.py:119-121 (per buffer) and the frame loop of
 * mlab.psd behind process_sigmf_data.py:188, batched over all frames of the input. */
SPX_API int spx_stft_exec(spx_plan* plan, spx_stft_args* args);

/* spx_stft_exec plus the persistence spectrum of the call's uint8 waterfall levels (counts[n_streams][256][nfft],
 * uint32, in args->mem space; args->accumulate applies to it as to welch_acc / maxhold).  args->wf_rows may be NULL:
 * the rows are then produced into plan-owned device scratch and never leave the GPU.
 *   counts[s][q][j] = number of frames f of stream s whose level wf_rows[s*F + f][j] is q, so every column sums to F.
 * Level q holds dB values in [vmin + q*D, vmin + (q+1)*D), D = (vmax - vmin)/256; level 0 also holds everything below
 * vmin and NaN, level 255 everything at or above vmax - D.  Needs vmax > vmin even without wf_rows; peer_outputs != 0
 * returns SPX_E_UNSUPPORTED.  Without caller rows, a device-resident call transforms the frames in batches through a
 * row buffer of SPX_PERSIST_ROWS_BYTES (plan-creation environment variable, default 64 MiB), and a host-memory call
 * copies back only the counts and the accumulators (d2h_bytes_out). */
SPX_API int spx_stft_exec_persistence(spx_plan* plan, spx_stft_args* args, uint32_t* counts);

/* Pooled spectrogram (display detectors).  Row g of stream s pools frames [gK, min((g+1)K, F_total)) and column c pools
 * bins [cB, (c+1)B) (fftshift order) of the power P = |X|^2 that the dB rows encode:
 *   SPX_POOL_MEAN: acc[s][g][c] = sum of P over the cell (NaN propagates, as in welch_acc)
 *   SPX_POOL_MAX:  acc[s][g][c] = max of the dB value over the cell (NaN skipped; -inf when nothing or only NaN)
 * The power is recovered from the float32 dB rows as (10^(d/20) - db_eps)^2, clipped at 0. */
#define SPX_POOL_MEAN 0
#define SPX_POOL_MAX 1

typedef struct {
    uint32_t struct_size;     /* sizeof(spx_pool_args) */
    int32_t mode;             /* SPX_POOL_* */
    int64_t frames_per_row;   /* K >= 1 */
    int32_t bins_per_col;     /* B >= 1, nfft % B == 0 */
    int32_t reserved;
    int64_t first_frame;      /* global index of this call's frame 0 (>= 0): calls on consecutive pieces of a capture
                                 pool into one accumulator, a row may span calls */
    int64_t n_rows;           /* G the accumulator holds; every frame of the call must fall in a row < G */
    double* acc;              /* [n_streams][G][nfft / B], args->mem space; args->accumulate applies (0: set to the mode's
                                 identity, 0 or -inf, before adding) */
} spx_pool_args;

/* spx_stft_exec plus the pooled accumulator of the call's frames.  args->db_rows may be NULL: the dB rows then go in
 * batches through a plan-owned float row buffer of SPX_POOL_ROWS_BYTES (plan-creation environment variable, default
 * 256 MiB) and never leave the GPU; a host-memory call then copies back only the accumulator, the other accumulators and
 * the rows that were asked for (d2h_bytes_out).  SPX_E_INVALID for K < 1, B < 1, nfft % B != 0, an unknown mode,
 * first_frame < 0 or a frame in a row >= n_rows; SPX_E_UNSUPPORTED for peer_outputs.  N = 65536 runs the two-kernel
 * four-step path (float rows). */
SPX_API int spx_stft_exec_pooled(spx_plan* plan, spx_stft_args* args, spx_pool_args* pool);

/* Pooled dB (db_out, float32) and/or levels (wf_out, uint8; needs vmax > vmin) of an accumulator, both
 * [n_streams][n_rows][nfft / B] in `mem` space:
 *   mean: 20 log10(sqrt(acc / (n_g B)) + db_eps), n_g = the frames of row g;   max: acc
 *   level = clip(floor((dB - vmin) * 256 / (vmax - vmin)), 0, 255), NaN -> 0, computed in float64 from the float32 dB.
 * n_rows must be ceil(n_frames_total / frames_per_row). */
SPX_API int spx_pool_finalize(spx_plan* plan, int32_t mem, int32_t mode, const double* acc, int32_t n_streams,
                              int64_t n_rows, int64_t n_frames_total, int64_t frames_per_row, int32_t bins_per_col,
                              float* db_out, uint8_t* wf_out, float vmin, float vmax, void* stream);

/* ---------------------------------------------------------------- digital down-converter (zoom)
 * Mixes a band of interest to 0 Hz with a 64-bit NCO, low-pass filters it and keeps every decim-th output, so that the
 * STFT path can look at a narrow band of a wide capture ("zoom").  For input x[n] (in_fmt samples times in_scale) whose
 * sample n has global index first_sample + n:
 *   phi(n) = ((first_sample + n) * phase_inc) mod 2^64              (exact integer arithmetic)
 *   mix[n] = x[n] * exp(-2 pi i phi(n) / 2^64)                      (tuned shift = phase_inc * fs / 2^64)
 *   y[m]   = sum_k h[k] mix[m D + T - 1 - k],  m = 0 .. M - 1,  M = (n_samples - T) / D + 1 (0 if n_samples < T)
 * i.e. numpy's convolve(mix, h, 'valid')[::D].  The output rate is fs / D and its centre frequency fc + shift; with odd
 * symmetric taps y[m] belongs to time (first_sample + m D + (T - 1) / 2) / fs.  Consecutive calls on pieces of a capture
 * that overlap by T - D samples, each with the global first_sample of its piece, give the outputs of one call bit for bit:
 * the arithmetic of y[m] depends only on global indices, the taps and the input.  Decimations beyond one stage (T > 8192)
 * are two DDCs in cascade, the second with phase_inc 0. */
typedef struct spx_ddc spx_ddc;

typedef struct {
    uint32_t struct_size;  /* sizeof(spx_ddc_config) */
    int32_t device;
    int32_t in_fmt;        /* SPX_FMT_* */
    float in_scale;        /* multiplies every sample (0 = 1.0) */
    int32_t decim;         /* D >= 1 (D > 2048 may return SPX_E_UNSUPPORTED: cascade two DDCs) */
    int32_t n_taps;        /* T in [1, 8192] */
    const double* taps;    /* host, h[0 .. T - 1]; rounded once to float32 at create */
    int64_t phase_inc;     /* round(shift_hz / fs * 2^64) as two's complement */
} spx_ddc_config;

SPX_API int spx_ddc_create(spx_ddc** out, const spx_ddc_config* cfg);
SPX_API int spx_ddc_destroy(spx_ddc* ddc);
/* wait for everything the handle has enqueued on its own streams */
SPX_API int spx_ddc_sync(spx_ddc* ddc);
/* y of n_samples samples into out[M][2] (float32 I, Q); *n_out = M.  SPX_MEM_DEVICE: `in` / `out` are device pointers
 * used on `stream` (NULL = the handle's stream), nothing is synchronised.  SPX_MEM_HOST: the input is staged through
 * pieces of SPX_H2D_PIECE_BYTES (handle-creation environment variable, default 16 MiB) cut at output boundaries, the
 * upload of one piece overlapping the kernel of the previous one; the call returns when `out` is written.  in and out
 * must be 4-byte aligned.  SPX_E_INVALID for a bad mem, n_samples < 0, first_sample < 0, or NULL in / out when M > 0. */
SPX_API int spx_ddc_exec(spx_ddc* ddc, int32_t mem, const void* in, int64_t n_samples, int64_t first_sample, float* out,
                         int64_t* n_out, int64_t* h2d_bytes_out, int64_t* d2h_bytes_out, void* stream);

/* Many down-conversions of one capture in one launch: each job is the DDC above with its own NCO and its own span, and all
 * share the handle's in_fmt, in_scale, taps (T) and decimation (D).  Job j computes
 *   y_j[m] = sum_k h[k] mix_j[first_sample_j + m D + T - 1 - k],   m = m0_j .. m0_j + n_out_j - 1
 * where mix_j uses phase_inc_j and the global sample index exactly as spx_ddc_exec does (the handle's own phase_inc is
 * not used), so y_j[m] has the bits of output m of spx_ddc_exec on a DDC with phase_inc_j called with
 * first_sample = first_sample_j. */
typedef struct {
    int64_t first_sample;  /* global index of the job's sample 0: its output m starts at first_sample + m*D */
    int64_t phase_inc;     /* the job's NCO, as spx_ddc_config.phase_inc */
    int64_t m0;            /* first output of the job written by this call */
    int64_t n_out;         /* outputs written by this call (0 allowed) */
    int64_t out_offset;    /* output m goes to out[out_offset + m - m0] (complex, float32 I,Q) */
} spx_ddc_job;

/* The jobs over `in` (device), whose sample 0 has global index in_first_sample, into `out` (device), enqueued on `stream`
 * (NULL = the handle's stream); nothing is synchronised.  `jobs` is host memory; it is copied to the device on `stream`
 * through a pinned staging buffer of the handle, and may be reused once the call returns.  Every window
 * [first_sample + m D, first_sample + m D + T) of a job must lie in [in_first_sample, in_first_sample + n_samples).
 * Columns of out that no job writes are left untouched.  The output regions of different jobs must not overlap; this is
 * not checked.  SPX_E_INVALID, with nothing launched, for n_samples, in_first_sample or n_jobs < 0, jobs NULL with
 * n_jobs > 0, a job with a negative first_sample, m0, n_out or out_offset, a window outside the input, or (when some job
 * has outputs) in or out NULL or not 4-byte aligned.  Jobs with n_out = 0 are skipped; a call without outputs launches
 * nothing. */
SPX_API int spx_ddc_exec_jobs(spx_ddc* ddc, const void* in, int64_t n_samples, int64_t in_first_sample,
                              const spx_ddc_job* jobs, int32_t n_jobs, float* out, void* stream);

/* ---------------------------------------------------------------- polyphase channelizer (channel scan)
 * Splits a wideband capture into M baseband channels in one pass: all M down-conversions of the DDC above at once.  With
 * the DDC's names (x = in_fmt samples times in_scale, sample n has global index first_sample + n, real taps h[0 .. T-1]),
 * channel j = 0 .. M-1 in fftshift order, offset c = j - M/2, is the DDC with phase_inc_j = c 2^64 / M (mod 2^64), taps h
 * and decimation D:
 *   y_j[m] = sum_k h[k] x[mD + T-1-k] exp(-2 pi i c (first_sample + mD + T-1-k) / M),   m = 0 .. n_out - 1
 *   n_out  = (n_samples - T) / D + 1   (0 if n_samples < T), as spx_ddc_exec
 * Channel j is centred at fc + c fs / M and runs at fs / D; a tone at its centre comes out at 0 Hz.  It is computed as a
 * fold of the taps by global sample class (first_sample + n) mod M followed by one M-point FFT per output step, and the
 * arithmetic of y_j[m] depends only on global indices, the taps and the input: calls on pieces of a capture that overlap
 * by T - D samples, each with the global first_sample of its piece, give the outputs of one call bit for bit.
 * Supported: M a power of two in [16, 4096]; D = M (critically sampled) or M / 2 (2x oversampled); T in [1, 32 M]. */
typedef struct spx_chan spx_chan;

typedef struct {
    uint32_t struct_size;  /* sizeof(spx_chan_config) */
    int32_t device;
    int32_t in_fmt;        /* SPX_FMT_* */
    float in_scale;        /* multiplies every sample (0 = 1.0) */
    int32_t n_channels;    /* M: power of two in [16, 4096] */
    int32_t decim;         /* D: M or M / 2 */
    int32_t n_taps;        /* T in [1, 32 M] */
    const double* taps;    /* host, h[0 .. T - 1]; rounded once to float32 at create */
} spx_chan_config;

/* SPX_E_INVALID: NULL out / cfg, a wrong struct_size, M not a power of two in [16, 4096], D not M or M / 2, T outside
 * [1, 32 M], NULL taps, an unknown in_fmt, a device index out of range.  SPX_E_NODEVICE: no CUDA device (no CPU
 * fallback). */
SPX_API int spx_chan_create(spx_chan** out, const spx_chan_config* cfg);
SPX_API int spx_chan_destroy(spx_chan* chan);
/* wait for everything the handle has enqueued on its own streams; SPX_E_INVALID for NULL */
SPX_API int spx_chan_sync(spx_chan* chan);
/* The channels of n_samples samples into out[M][out_stride] (complex64 as float32 I, Q; channel-major, columns
 * n_out .. out_stride - 1 are left as they are); *n_out = n_out.  SPX_MEM_DEVICE: `in` / `out` are device pointers used
 * on `stream` (NULL = the handle's stream), nothing is synchronised.  SPX_MEM_HOST: the input is staged through pieces
 * of SPX_H2D_PIECE_BYTES (handle-creation environment variable, default 16 MiB) cut at output boundaries with the T - D
 * halo; each piece's [M][per] block is copied into the host rows as it finishes, and the call returns when `out` is
 * written.  SPX_E_INVALID for a NULL handle, a bad mem, n_samples < 0, first_sample < 0, and, when n_out > 0,
 * out_stride < n_out, NULL in or out, `in` not 4-byte or `out` not 8-byte aligned.  n_out = 0 launches nothing. */
SPX_API int spx_chan_exec(spx_chan* chan, int32_t mem, const void* in, int64_t n_samples, int64_t first_sample,
                          float* out, int64_t out_stride, int64_t* n_out, int64_t* h2d_bytes_out, int64_t* d2h_bytes_out,
                          void* stream);

/* Measurement helper: runs spx_stft_exec (SPX_MEM_DEVICE buffers only) warmup+iters times on the
 * launch stream, each bracketed by CUDA events; optionally READS a 256 MiB buffer before every
 * iteration to flush the 126 MB L2 without leaving dirty lines behind.  ms_each[iters] receives the device time of
 * each timed launch. */
SPX_API int spx_stft_time(spx_plan* plan, spx_stft_args* args, int32_t warmup, int32_t iters, int32_t flush_l2,
                          float* ms_each);

/* Welch density from the accumulated numerator: Pxx[k] = acc[k] / (n_frames * fs * sum(w^2))
 * (mlab.psd, two-sided) and 10*log10 of it.  Either output may be NULL.  `mem` as above. */
SPX_API int spx_welch_finalize(spx_plan* plan, int32_t mem, const double* welch_acc, int64_t n_frames, double fs,
                       double* pxx, double* pxx_db, void* stream);

/* The same for `n_streams` accumulators laid out [n_streams][nfft] (one launch; every stream has n_frames frames). */
SPX_API int spx_welch_finalize_batch(spx_plan* plan, int32_t mem, const double* welch_acc, int32_t n_streams,
                                     int64_t n_frames, double fs, double* pxx, double* pxx_db, void* stream);

/* The plan's compute stream (cudaStream_t), so that callers can order their own SPX_MEM_DEVICE calls
 * (spx_welch_finalize, spx_classify_features, spx_timer_*) after the plan's kernels. */
SPX_API int spx_plan_stream(spx_plan* plan, void** stream_out);

/* Device-side stopwatch: a pair of CUDA events recorded on `stream` (NULL = the legacy default stream).
 * spx_timer_elapsed_ms waits for the stop event.  Used by bench.py to time K steps on the launching stream. */
typedef struct spx_timer spx_timer;
SPX_API int spx_timer_create(int32_t device, spx_timer** out);
SPX_API int spx_timer_start(spx_timer* t, void* stream);
SPX_API int spx_timer_stop(spx_timer* t, void* stream);
SPX_API int spx_timer_elapsed_ms(spx_timer* t, float* ms_out);
SPX_API int spx_timer_destroy(spx_timer* t);

/* sum(w^2) and sum(w) of the plan's float64 window (in_scale is applied to the data, not counted here) */
SPX_API int spx_plan_window_sums(spx_plan* plan, double* sum_w2, double* sum_w);

/* ---------------------------------------------------------------- classifier measurements */
/* What classify_signal_advanced / classify_signal_simple measure on one spectrum
 * (/root/reference/app/processing/classifier.py:45-58 and :18-23; helpers :163-219).
 * Bin indices are exact; the host layer turns them into Hz with the caller's `freqs` array and
 * applies the label rules + temporal smoothing (:60-161).
 * Non-finite bins follow numpy: NaN (either sign bit) is the maximum and sorts after +inf; every comparison
 * with a NaN threshold is false, so a NaN peak gives no edges and no peaks; ±inf enter the sums as numpy's do. */
typedef struct {
    int32_t n;                 /* bins */
    int32_t argmax;            /* np.argmax: the first NaN if any, else the first index of the maximum (0 for all -inf) */
    double peak_db;            /* np.max(power_db) (:46): NaN if any bin is NaN */
    double noise_floor_db;     /* np.percentile(power_db, 20), 'linear' (:181): NaN if any bin is NaN; numpy's lerp
                                  otherwise, so inf - inf inside it (e.g. all -inf, or n == 1 and infinite) is NaN */
    double snr_db;             /* peak - noise floor (:46), un-rounded */
    double adaptive_thr;       /* max(nf + 5, peak - 0.9 snr + 5) (:53) with Python's max: nf + 5 unless the second
                                  term is greater, so a NaN second term (one +inf bin) leaves nf + 5 */
    double p20_lo, p20_hi;     /* the two order statistics the percentile interpolates, NaN sorted last */
    int32_t min_distance_bins; /* max(3, n // 300) (:54) */
    int32_t first_3db, last_3db;   /* first/last bin with p >= peak - 3  (:163-170); -1 if none */
    int32_t first_10db, last_10db;
    int32_t first_20db, last_20db;
    int32_t simple_first, simple_last; /* first/last bin with p > peak - 20 (strict, :18-21) */
    double flatness;           /* exp(mean(ln p)) / mean(p), p = max(10^(dB/10), 1e-15), clipped to [0,1] (:183-189) */
    double kurtosis;           /* mean(((x - mu)/sigma)^4), 0 if sigma < 1e-9 (:191-198); NaN if sigma is NaN */
    double mean_db, std_db;
    int32_t n_candidates;      /* strict local maxima above adaptive_thr */
    int32_t peak_count;        /* after greedy min-distance thinning (:200-212) */
    double peak_spacing_std_bins; /* population std of successive peak spacings in bins (0 if < 3 peaks) */
    int32_t peaks_stored;      /* how many peak indices were written to `peaks` */
    int32_t reserved;
} spx_features;

/* optional overrides (NULL = the reference's choices: drops 3/10/20 dB, adaptive threshold, auto distance) */
typedef struct {
    double drop_db[3];           /* occupied-bandwidth drops reported in first/last_{3,10,20}db */
    double peak_threshold_db;    /* used when use_peak_threshold != 0 (classifier.py:200 `threshold_db`) */
    int32_t use_peak_threshold;
    int32_t min_distance_bins;   /* > 0 overrides max(3, n // 300) */
} spx_feature_opts;

/* power_db: `batch` spectra of n values (dtype 0 = float32, 1 = float64), spectrum b at b*stride.
 * out[batch] and peaks[batch][peaks_cap] (optional) are HOST buffers in both memory modes; the call
 * returns after the results have landed.  n == 0 yields zeroed features ("No Data"). */
SPX_API int spx_classify_features(int32_t device, int32_t mem, const void* power_db, int32_t dtype, int32_t n,
                                  int32_t batch, int64_t stride, spx_features* out, int32_t* peaks,
                                  int32_t peaks_cap, const spx_feature_opts* opts, void* stream);

/* Enqueue-only variant for pipelines that must not stall the host: device input, device output (`out_dev[batch]`,
 * optional `peaks_dev[batch][peaks_cap]`), nothing is copied or synchronised.  Pair it with spx_memcpy_d2h_async
 * into pinned memory and read the results after the stream has been synchronised. */
SPX_API int spx_classify_features_dev(int32_t device, const void* power_db_dev, int32_t dtype, int32_t n, int32_t batch,
                                      int64_t stride, spx_features* out_dev, int32_t* peaks_dev, int32_t peaks_cap,
                                      const spx_feature_opts* opts, void* stream);

/* ---------------------------------------------------------------- signal detection (regions of a dB image)
 * For a float32 dB image db[rows][cols] (row r at db + r * stride; a row is one time slice, columns in fftshift order):
 *   floor[r]   = np.percentile(float64(db[r]), 20): spx_features.noise_floor_db of the row, with its NaN rules (a row
 *                holding a NaN, or all -inf, has a NaN floor)
 *   mask[r][c] = float64(db[r][c]) >= floor[r] + threshold_db, compared in float64 (false for NaN cells and NaN floors)
 *   regions    = scipy.ndimage.label(mask, structure=np.ones((3, 3))): 8-connected, numbered in raster order of their
 *                first cell; regions of fewer than min_cells cells are dropped and the rest renumbered 1 .. n in that order
 * Every field below except power_sum, the labels and the floors are exact and identical from run to run. */
typedef struct {
    int32_t row0, row1, col0, col1;   /* inclusive bounding box */
    int64_t n_cells;                  /* cells in the region */
    int32_t peak_row, peak_col;       /* the cell of the largest dB; ties -> smallest raster index (r * cols + c) */
    double peak_db, peak_floor_db;    /* db at the peak (as float64); peak_floor_db = floor[peak_row] */
    double power_sum;                 /* sum of 10^(dB/10) over the region's cells, float64, accumulated with float64
                                         atomics: within ~1e-12 relative of an exact sum, but not bit-reproducible */
} spx_region;

/* Labels the regions of one image (K11).  `db` and the optional outputs `labels` (int32 [rows][cols]: region number
 * 1 .. n, 0 for cells outside every kept region) and `row_floor_db` (float64 [rows]) are in `mem` space; `regions` and
 * `n_regions_out` are HOST buffers in both memory modes, and the call returns after they have landed.  *n_regions_out =
 * the total n; the first min(n, max_regions) regions, in numbering order, go to regions[].  SPX_MEM_DEVICE work runs on
 * `stream` (NULL = the library's stream of the device).  rows == 0 or cols == 0: zero regions.
 * SPX_E_INVALID: a bad device or mem; negative rows or cols; rows * cols > INT32_MAX (checked before anything is
 * allocated); stride < cols; min_cells < 1; max_regions < 0; NULL db or n_regions_out; NULL regions with max_regions > 0.
 * SPX_E_NODEVICE without a CUDA device. */
SPX_API int spx_detect_regions(int32_t device, int32_t mem, const float* db, int32_t rows, int32_t cols, int64_t stride,
                               double threshold_db, int32_t min_cells, spx_region* regions, int32_t max_regions,
                               int32_t* n_regions_out, int32_t* labels, double* row_floor_db, void* stream);

/* ---------------------------------------------------------------- time-domain / constellation views */
/* 2-D I/Q density histogram with np.histogram2d(I, Q, bins, range=[[-R,R],[-R,R]]) semantics
 * (SURVEY.md A10; replaces the 2000-point scatter of app/dashboard/callbacks.py:199-214).
 * hist is uint32 [bins][bins], H[i][j] with i <-> I, j <-> Q; right edge inclusive, values outside
 * dropped; samples are multiplied by in_scale first.  accumulate != 0 adds to the existing counts. */
SPX_API int spx_iq_hist2d(int32_t device, int32_t mem, const void* in, int32_t in_fmt, double in_scale, int64_t n,
                          double r, int32_t bins, uint32_t* hist, int32_t accumulate, void* stream);

/* per-frame mean and peak of I^2+Q^2 (SURVEY.md A9; scripts/pyad-iio-test.py:93 prints the mean per
 * buffer); frames as in spx_frame_count(n, frame_len, hop); outputs float32 [F] each.  Non-finite powers follow
 * numpy's mean and max: when any I^2+Q^2 of a frame is NaN, its mean_pow and peak_pow are both NaN (the peak does not
 * skip NaN); otherwise an infinite power makes both +inf. */
SPX_API int spx_frame_stats(int32_t device, int32_t mem, const void* in, int32_t in_fmt, float in_scale, int64_t n,
                            int32_t frame_len, int32_t hop, float* mean_pow, float* peak_pow, int64_t* n_frames_out,
                            void* stream);

/* ---------------------------------------------------------------- streaming ingest: pinned ring */
/* Replaces the reference's queue of per-buffer dicts (app/sdr/streamer.py:18,123-131,186-200) for
 * high-rate ingest: the producer fills page-locked slots in place; spx_ring_commit enqueues
 * H2D -> fused STFT -> D2H on three streams and returns at once, so copies of slot k+1 overlap the
 * kernel of slot k.  Frames run continuously across slots (the unconsumed tail is carried on the device).
 * Every slot is one Welch / max-hold block.  The ring borrows the plan (keep it alive, same thread rules). */
typedef struct spx_ring spx_ring;

typedef struct {
    uint32_t struct_size;
    int32_t n_slots;        /* 2 .. 64 */
    int64_t slot_samples;   /* capacity of one slot, >= nfft */
    int32_t want_wf_rows, want_db_rows, want_welch, want_maxhold;
    float vmin, vmax;
    int32_t want_features;  /* per slot: Welch PSD in dB (mlab.psd normalisation with sample_rate) + the classifier
                             * measurements of it (classifier.py:45-58), computed on the device right behind the STFT
                             * kernel; needs want_welch */
    int32_t reserved;
    double sample_rate;     /* Fs of the PSD normalisation (want_features) */
} spx_ring_config;

typedef struct {
    uint32_t struct_size;
    int32_t reserved;
    int64_t seq;            /* commit sequence number of this slot */
    int64_t n_frames;       /* frames completed by this slot */
    int64_t first_frame;    /* global index of its first frame */
    const uint8_t* wf_rows; /* pinned host, [n_frames][nfft] (NULL if not requested) */
    const float* db_rows;
    const double* welch_acc;
    const float* maxhold;
    int64_t h2d_bytes, d2h_bytes; /* bytes this slot moved over PCIe, each direction */
    const double* pxx_db;         /* pinned host, [nfft] 10*log10 of the slot's Welch density (want_features) */
    const spx_features* features; /* pinned host, measurements of pxx_db (want_features) */
} spx_ring_result;

typedef struct {
    uint32_t struct_size;
    int32_t in_flight;
    int64_t h2d_bytes, d2h_bytes, samples, frames; /* totals since creation */
    int64_t reserved;
} spx_ring_stats_t;

SPX_API int spx_ring_create(spx_ring** out, spx_plan* plan, const spx_ring_config* cfg);
SPX_API int spx_ring_destroy(spx_ring* ring);
/* next pinned slot to fill; SPX_E_BUSY when all slots are in flight / unreleased */
SPX_API int spx_ring_acquire(spx_ring* ring, void** host_slot, int64_t* capacity_samples);
/* the acquired slot now holds n_samples samples: enqueue its copies and kernel (does not block) */
SPX_API int spx_ring_commit(spx_ring* ring, int64_t n_samples);
/* wait for the oldest committed slot and expose its (pinned) results; they stay valid until release */
SPX_API int spx_ring_collect(spx_ring* ring, spx_ring_result* out);
SPX_API int spx_ring_release(spx_ring* ring);
SPX_API int spx_ring_stats(spx_ring* ring, spx_ring_stats_t* out);

#ifdef __cplusplus
}
#endif
#endif /* SPX_H_ */
