/*
 * b200dsp.h -- C-ABI of libb200dsp.so: the B200 (sm_100a) implementation of the
 * newsched data-parallel block hot path.
 *
 * This is the drop-in boundary (SURVEY.md 8b).  Every entry point is `extern "C"`, takes
 * plain pointers and sizes (device pointers unless the name says `_host`), returns an int
 * status (0 = ok, < 0 = error, text via b200_last_error()), never allocates or
 * synchronises inside a `_run` call, and launches on the caller's stream.  The host-side
 * C++17 block wrappers (include/gnuradio/blocklib/cuda/ *.hpp) and the Python mirror
 * (newsched_b200/) are thin shims over exactly these symbols.
 *
 * Each op lists the reference interface it stands behind:
 *   copy            gr::blocks::copy::work         blocklib/blocks/include/gnuradio/blocklib/blocks/copy.hpp:33-44
 *                   gr::cuda::copy::work           blocklib/cuda/lib/copy.cpp:41-63 (+ copy.cu:6-28)
 *   multiply_const  gr::blocks::multiply_const<T>  blocklib/blocks/lib/multiply_const.cpp:19-81
 *                   gr::cuda::multiply_const       blocklib/cuda/lib/multiply_const.cpp:9-16 (+ .cu:1-17)
 *   ring            gr::cuda_buffer                runtime/include/gnuradio/cudabuffer.hpp:34-79, runtime/lib/cudabuffer.cu:17-183
 *   fir / fft / complex_to_mag / pfb_channelizer   absent from the reference snapshot (SURVEY.md 0.1);
 *                   the work() contract is gr::block::work, runtime/include/gnuradio/block.hpp:81-85,
 *                   semantics fixed in SURVEY.md 8(c).
 */
#ifndef B200DSP_H
#define B200DSP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B200_API __attribute__((visibility("default")))
#else
#define B200_API
#endif

/* opaque; layout-compatible with cudaStream_t / cudaEvent_t */
typedef struct CUstream_st* b200_stream_t;
typedef struct CUevent_st* b200_event_t;

enum {
    B200_OK = 0,
    B200_ERR_ARG = -1,     /* bad argument (null handle, size, alignment, unsupported N ...) */
    B200_ERR_CUDA = -2,    /* a CUDA runtime / driver call failed */
    B200_ERR_NOMEM = -3,   /* allocation failed */
    B200_ERR_UNSUPPORTED = -4
};

/* ---- library / device ----------------------------------------------------------- */
B200_API int b200_version(void);                 /* major*10000 + minor*100 + patch */
B200_API const char* b200_last_error(void);      /* thread-local text of the last failure */
B200_API int b200_device_count(int* count);
B200_API int b200_set_device(int device);
B200_API int b200_get_device(int* device);
B200_API int b200_device_sm_count(int* sms);
B200_API int b200_device_synchronize(void);
B200_API int64_t b200_launch_count(void);        /* kernels launched by this library so far (process-wide) */
/* measurement helper: runs a pure-FFMA kernel (iters x 256 FFMA per thread, 8 CTAs/SM) and
 * reports the FP32 FMA rate in TFLOP/s -- the denominator of the FP32-bound FIR roofline. */
B200_API int b200_measure_fp32_tflops(int iters, float* tflops, float* ms);
/* same probe written with the packed fma.rn.f32x2 (FFMA2) form that the FIR kernel uses */
B200_API int b200_measure_fp32x2_tflops(int iters, float* tflops, float* ms);

/* ---- memory / stream / event plumbing (so hosts need no CUDA headers) ------------ */
B200_API int b200_malloc(void** dptr, size_t bytes);
B200_API int b200_free(void* dptr);
B200_API int b200_host_alloc(void** hptr, size_t bytes);   /* pinned */
B200_API int b200_host_free(void* hptr);
B200_API int b200_host_register(void* hptr, size_t bytes); /* pin an existing allocation */
B200_API int b200_host_unregister(void* hptr);
B200_API int b200_memcpy_h2d(void* dst, const void* src, size_t bytes, b200_stream_t s);
B200_API int b200_memcpy_d2h(void* dst, const void* src, size_t bytes, b200_stream_t s);
B200_API int b200_memcpy_d2d(void* dst, const void* src, size_t bytes, b200_stream_t s);
B200_API int b200_memset(void* dst, int value, size_t bytes, b200_stream_t s);
B200_API int b200_stream_create(b200_stream_t* s);
B200_API int b200_stream_destroy(b200_stream_t s);
B200_API int b200_stream_synchronize(b200_stream_t s);
B200_API int b200_stream_activate(b200_stream_t s);        /* current device := the stream's device */
B200_API int b200_stream_wait_event(b200_stream_t s, b200_event_t e);
B200_API int b200_event_create(b200_event_t* e, int timing);
B200_API int b200_event_destroy(b200_event_t e);
B200_API int b200_event_record(b200_event_t e, b200_stream_t s);
B200_API int b200_event_synchronize(b200_event_t e);
B200_API int b200_event_query(b200_event_t e);             /* 0 = complete, 1 = not yet, <0 error */
B200_API int b200_event_elapsed_ms(b200_event_t start, b200_event_t stop, float* ms);

/* ---- peer memory (SURVEY.md 8e: time-segment sharding needs the (ntaps-1)-sample halo that precedes
 * a GPU's segment, which lives at the end of the left neighbour's segment).  Instead of exchanging it,
 * the neighbour's buffer is mapped into this GPU's address space and the FIR / channelizer kernels read
 * the halo straight over NVLink (`d_halo` of the *_run_segment calls may be such a pointer).
 * One process, several devices: b200_enable_peer_access(peer) on the current device.
 * One process per device: export a handle for any pointer inside a cudaMalloc allocation, ship the
 * 88 bytes to the other process (any host channel), import it there.  The reference has no multi-device
 * concept (SURVEY.md 5); its edges are created per flowgraph in one process,
 * schedulers/mt/lib/buffer_management.cpp:78-82. */
typedef struct {
    unsigned char bytes[64]; /* cudaIpcMemHandle_t of the allocation */
    uint64_t offset;         /* of the exported pointer inside the allocation */
    uint64_t size;           /* of the allocation */
    int32_t device;          /* exporting device ordinal (as that process numbers it) */
    int32_t reserved;
} b200_ipc_handle;
B200_API int b200_enable_peer_access(int peer_device);
B200_API int b200_ipc_export(const void* dptr, b200_ipc_handle* out);
B200_API int b200_ipc_import(const b200_ipc_handle* h, void** dptr);
B200_API int b200_ipc_close(const b200_ipc_handle* h, void* dptr);

/* ---- device-resident doubly mapped ring (replaces gr::cuda_buffer, cudabuffer.cu:17-183)
 * One physical allocation of `size` bytes mapped twice back to back with the CUDA VMM API,
 * so base[i] and base[i + size] alias: any window of <= size bytes starting anywhere in
 * [base, base+size) is linearly addressable, with no mirror copies (the reference emulates
 * this with 1-3 cudaMemcpyAsync + a stream sync per post_write, cudabuffer.cu:116-176).
 * `min_bytes` is rounded up to the allocation granularity; the result is in *size. */
typedef struct b200_ring b200_ring;
B200_API int b200_ring_create(size_t min_bytes, b200_ring** ring);
B200_API int b200_ring_destroy(b200_ring* ring);
B200_API int b200_ring_enable_peer(b200_ring* ring, int peer_device); /* grant another GPU access to the ring */
B200_API void* b200_ring_base(const b200_ring* ring);
B200_API size_t b200_ring_size(const b200_ring* ring);
B200_API size_t b200_ring_granularity(void);

/* ---- elementwise stream blocks ---------------------------------------------------
 * copy: bit-exact byte copy of n_bytes (any alignment).  copy.hpp:33-44. */
B200_API int b200_copy(void* d_out, const void* d_in, size_t n_bytes, b200_stream_t s);
/* multiply_const over n scalars (n = n_items * vlen), multiply_const.cpp:19-81.
 * cc: out = in * (k_re + j k_im), products rounded to fp32 then added (no FMA), the
 * non-fused VOLK generic-kernel arithmetic. */
B200_API int b200_multiply_const_ff(float* d_out, const float* d_in, float k, size_t n, b200_stream_t s);
B200_API int b200_multiply_const_cc(void* d_out, const void* d_in, float k_re, float k_im, size_t n, b200_stream_t s);
B200_API int b200_multiply_const_ss(int16_t* d_out, const int16_t* d_in, int16_t k, size_t n, b200_stream_t s);
B200_API int b200_multiply_const_ii(int32_t* d_out, const int32_t* d_in, int32_t k, size_t n, b200_stream_t s);
/* two-input stream blocks (SURVEY.md 8f rank 4: natural neighbours on the same kernels):
 * out = a * b / out = a + b over n scalars; cc = full complex product, non-fused rounding. */
B200_API int b200_multiply_ff(float* d_out, const float* d_a, const float* d_b, size_t n, b200_stream_t s);
B200_API int b200_multiply_cc(void* d_out, const void* d_a, const void* d_b, size_t n, b200_stream_t s);
B200_API int b200_add_ff(float* d_out, const float* d_a, const float* d_b, size_t n, b200_stream_t s);
B200_API int b200_add_cc(void* d_out, const void* d_a, const void* d_b, size_t n, b200_stream_t s);
/* complex_to_mag: out[i] = sqrtf(re*re + im*im) over n complex64 (SURVEY.md 8c). */
B200_API int b200_complex_to_mag(float* d_out, const void* d_in, size_t n, b200_stream_t s);
B200_API int b200_complex_to_mag_squared(float* d_out, const void* d_in, size_t n, b200_stream_t s);

/* ---- fir_filter (ccf: complex64 stream, real taps; fff: float stream) -------------
 * y[m] = sum_{k<T} h[k] x[m*D - k], decimation phase 0, m = 0 .. floor(n_in/D)-1.
 * The handle owns the (T-1)-sample history that precedes the next input item (zeros at
 * creation), so a stream may be fed in arbitrary chunks: each run consumes
 * n_consumed = n_produced*D items and leaves n_in % D items for the caller to re-present.
 * An optional fused epilogue multiplies every output by a complex (ccf) / real (fff)
 * constant -- the adjacent multiply_const of BASELINE config 3. */
typedef struct b200_fir b200_fir;
typedef struct {
    const float* taps;    /* host pointer, n_taps floats */
    int32_t n_taps;
    int32_t decimation;   /* >= 1 */
    int32_t is_complex;   /* 1 = ccf, 0 = fff */
    int32_t fuse_multiply_const; /* 0/1 */
    float k_re, k_im;     /* epilogue constant (k_im ignored for fff) */
    int32_t algorithm;    /* 0 = auto, 1 = direct SIMT, 2 = block-Toeplitz GEMM on the tensor cores (tcgen05; ccf with D <= 8, fff with D = 1 and <= 449 taps), 3 = overlap-save FFT,
                             4 = one thread per output (fallback); any other value is rejected with B200_ERR_ARG */
} b200_fir_params;
B200_API int b200_fir_create(const b200_fir_params* p, b200_fir** h);
B200_API int b200_fir_destroy(b200_fir* h);
B200_API int b200_fir_run(b200_fir* h, const void* d_in, void* d_out, int64_t n_in_items,
                          int64_t* n_consumed, int64_t* n_produced, b200_stream_t s);
/* stateless form for time-segment sharding: d_in points at the first NEW sample and the
 * T-1 samples before it are read from d_halo (device; NULL = zeros); handle state untouched. */
B200_API int b200_fir_run_segment(b200_fir* h, const void* d_halo, const void* d_in, void* d_out,
                                  int64_t n_in_items, int64_t* n_produced, b200_stream_t s);
B200_API int b200_fir_reset(b200_fir* h, b200_stream_t s);              /* history := zeros */
B200_API int b200_fir_set_history(b200_fir* h, const void* d_hist, b200_stream_t s); /* T-1 items, oldest first */
B200_API int b200_fir_get_history(b200_fir* h, void* d_hist, b200_stream_t s);
B200_API int b200_fir_algorithm(const b200_fir* h);                     /* what auto selected */
B200_API int b200_fir_geometry(const b200_fir* h, int* decimation, int* item_bytes);

/* ---- interp_fir_filter / rational_resampler (ccf / fff; SURVEY.md 8(f) row 4) ------
 * y[m] = sum_k h[k] xu[m*D - k] with xu = x zero-stuffed by L (polyphase: only the T/L products
 * per output that meet a real sample are formed).  interpolation L, decimation D; D = 1 is
 * interp_fir_filter.  A run consumes whole groups of D items and produces L per group
 * (n_consumed = floor(n_in/D)*D, n_produced = floor(n_in/D)*L), so every call starts at phase 0;
 * the ceil(T/L)-1 input samples of history live in the handle.  Absent from the reference
 * snapshot; the block interface it stands behind is gr::block::work
 * (runtime/include/gnuradio/block.hpp:81-85). */
typedef struct b200_resampler b200_resampler;
typedef struct {
    const float* taps;     /* host pointer, n_taps floats */
    int32_t n_taps;
    int32_t interpolation; /* L >= 1 */
    int32_t decimation;    /* D >= 1 */
    int32_t is_complex;    /* 1 = ccf, 0 = fff */
} b200_resampler_params;
B200_API int b200_resampler_create(const b200_resampler_params* p, b200_resampler** h);
B200_API int b200_resampler_destroy(b200_resampler* h);
B200_API int b200_resampler_run(b200_resampler* h, const void* d_in, void* d_out, int64_t n_in_items,
                                int64_t* n_consumed, int64_t* n_produced, b200_stream_t s);
/* stateless: the ceil(T/L)-1 samples before d_in[0] come from d_halo (device; NULL = zeros) */
B200_API int b200_resampler_run_segment(b200_resampler* h, const void* d_halo, const void* d_in, void* d_out,
                                        int64_t n_in_items, int64_t* n_produced, b200_stream_t s);
B200_API int b200_resampler_reset(b200_resampler* h, b200_stream_t s);
B200_API int b200_resampler_geometry(const b200_resampler* h, int* interpolation, int* decimation,
                                     int* item_bytes);

/* ---- fft (vector length N, forward / reverse, optional window, optional shift) -----
 * fft_vcc semantics (SURVEY.md 8c); no 1/N scaling.  Shared-memory Stockham, no cuFFT.
 * Prologue fusion: an adjacent upstream multiply_const_cc (pre_scale).
 * Epilogue fusion: an adjacent downstream complex_to_mag / mag_squared (output float32). */
typedef struct b200_fft b200_fft;
enum { B200_FFT_OUT_COMPLEX = 0, B200_FFT_OUT_MAG = 1, B200_FFT_OUT_MAG_SQUARED = 2 };
typedef struct {
    int32_t n;             /* power of two, 8 .. 8192 */
    int32_t forward;       /* 1 = forward (e^-j), 0 = reverse (e^+j) */
    const float* window;   /* host pointer, n floats, or NULL */
    int32_t shift;         /* fftshift of the output (forward) / ifftshift of the input (reverse) */
    int32_t output;        /* B200_FFT_OUT_* */
    int32_t fuse_pre_multiply_const; /* 0/1: x := x * (k_re + j k_im) before the window */
    float k_re, k_im;
} b200_fft_params;
B200_API int b200_fft_create(const b200_fft_params* p, b200_fft** h);
B200_API int b200_fft_destroy(b200_fft* h);
B200_API int b200_fft_run(b200_fft* h, const void* d_in, void* d_out, int64_t n_vectors, b200_stream_t s);
B200_API int b200_fft_geometry(const b200_fft* h, int* n, int* out_item_bytes);

/* ---- polyphase channelizer (analysis bank, M channels, critically sampled or oversampled) ----------
 * SURVEY.md 8(c): taps h[0..M*P), u_i[t] = sum_r h[i+rM] x[(t-r)M + M-1-i],
 * y_c[t] = sum_i u_i[t] e^{+j 2 pi i c / M}; out[t*M + c].  Handle keeps (P-1)*M history.
 * channel_begin/channel_count select a slice of output channels (channel sharding);
 * out is then [t][channel_count].
 *
 * oversample OS = 2 or 4 (GNU Radio's pfb_channelizer_ccf oversample_rate): one frame per hop D = M/OS input
 * samples, so adjacent channels overlap and a signal on a channel boundary is whole in both.  With t the frame
 * index since creation or the last reset (input before the stream start is zero):
 *   z_c[t] = e^{-j 2 pi c tD/M} sum_{n<MP} h[n] e^{+j 2 pi n c/M} x[tD + D-1-n]
 *          = sum_{i<M} u_{(i + tD) mod M}[t] e^{+j 2 pi i c/M},  u_i[t] = sum_r h[i+rM] x[tD + D-1-i-rM]
 * Every channel is at baseband (a tone at c0 fs/M is a constant phasor in channel c0).  OS = 1 is the formula
 * above.  A run consumes n_frames*D items and produces n_frames = floor(n_in/D) vectors; the handle keeps the
 * last P*M - D input samples and the frame phase (frames produced mod OS); b200_pfb_reset zeroes both.
 * b200_pfb_run_segment is stateless: d_halo holds the P*M - D samples before d_in (NULL = zeros) and d_in[0]
 * starts frame phase 0, so segments meant to join into one stream must start at multiples of M input samples
 * (e.g. multigpu.time_segments(..., align=M)).
 * OS > 1 needs M in 16..256 and the single-pass kernel (P up to its shared-memory limit; B200_ERR_UNSUPPORTED
 * otherwise), and the SIMT DFT (algorithm 2 is refused with B200_ERR_UNSUPPORTED). */
typedef struct b200_pfb b200_pfb;
typedef struct {
    const float* taps;   /* host, M*P floats */
    int32_t n_channels;  /* M, power of two 4..256 */
    int32_t taps_per_channel; /* P */
    int32_t channel_begin;
    int32_t channel_count; /* 0 = all */
    int32_t oversample;    /* 0 or 1 = critically sampled; 2, 4 = oversampled; anything else: B200_ERR_ARG */
} b200_pfb_params;
B200_API int b200_pfb_create(const b200_pfb_params* p, b200_pfb** h);
B200_API int b200_pfb_destroy(b200_pfb* h);
B200_API int b200_pfb_run(b200_pfb* h, const void* d_in, void* d_out, int64_t n_in_items,
                          int64_t* n_consumed, int64_t* n_produced_vectors, b200_stream_t s);
B200_API int b200_pfb_run_segment(b200_pfb* h, const void* d_halo, const void* d_in, void* d_out,
                                  int64_t n_in_items, int64_t* n_produced_vectors, b200_stream_t s);
B200_API int b200_pfb_reset(b200_pfb* h, b200_stream_t s);
B200_API int b200_pfb_geometry(const b200_pfb* h, int* n_channels, int* channel_count);
/* Form of the M = 64 channelizer (BASELINE.json configs[3] "filterbank + DFT as tensor-core GEMM"):
 *   0 = auto (the faster one as measured, DESIGN.md 4.4), 1 = branch filters + 64-point DFT on the SIMT pipes,
 *   2 = branch filters on the SIMT pipes, the DFT across branches as a 128 x 64 x 128 bf16-split GEMM per
 *       64-frame tile on tcgen05 with the DFT matrix resident in tensor memory (64 channels, <= 16 taps per
 *       channel; B200_ERR_UNSUPPORTED otherwise).  Same results within the 1e-5 relative-RMS bar. */
B200_API int b200_pfb_set_algorithm(b200_pfb* h, int32_t algorithm);
B200_API int b200_pfb_get_algorithm(const b200_pfb* h, int32_t* algorithm);
B200_API int b200_pfb_get_oversample(const b200_pfb* h, int32_t* oversample); /* 1, 2 or 4 */

/* ---- host-buffer streaming driver (the e2e path a host-resident source/sink sees) ---
 * A chain is an ordered list of op handles executed back to back on device buffers; the
 * `_run_host` call streams a HOST input through it in chunks with H2D / compute / D2H
 * overlapped on three streams and writes the HOST output.  Adjacent elementwise ops are
 * fused by the caller when building the handles (see fuse_* fields above). */
typedef struct b200_chain b200_chain;
enum { B200_OP_COPY = 1, B200_OP_MULTIPLY_CONST_CC = 2, B200_OP_COMPLEX_TO_MAG = 3,
       B200_OP_FIR = 4, B200_OP_FFT = 5, B200_OP_PFB = 6, B200_OP_MULTIPLY_CONST_FF = 7 };
typedef struct {
    int32_t kind;        /* B200_OP_* */
    void* handle;        /* b200_fir* / b200_fft* / b200_pfb* or NULL for stateless ops */
    float k_re, k_im;    /* multiply_const constant */
} b200_chain_op;
B200_API int b200_chain_create(const b200_chain_op* ops, int32_t n_ops, int32_t in_item_bytes,
                               int64_t chunk_items, b200_chain** c);
B200_API int b200_chain_destroy(b200_chain* c);
/* device-resident run: one pass over n_in_items already in HBM. */
B200_API int b200_chain_run(b200_chain* c, const void* d_in, void* d_out, int64_t n_in_items,
                            int64_t* n_out_bytes, b200_stream_t s);
/* host-resident run (blocking): h_in / h_out should be pinned for full PCIe rate. */
B200_API int b200_chain_run_host(b200_chain* c, const void* h_in, void* h_out, int64_t n_in_items,
                                 int64_t* n_out_bytes);
B200_API int64_t b200_chain_out_bytes_bound(const b200_chain* c, int64_t n_in_items);

#ifdef __cplusplus
}
#endif
#endif /* B200DSP_H */
