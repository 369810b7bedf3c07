/*
 * b200comms.h -- the drop-in boundary of the B200-native /comms/fir_filter + /comms/fft path.
 *
 * A plain C ABI: opaque handles, pointers and sizes, int status returns (0 = ok, <0 = error,
 * text via b200c_last_error()).  No exceptions, STL or torch types cross it.  The C++ block
 * layer (pothoscomms_b200/blocks/) is the only intended caller inside a Pothos process; the
 * Python ctypes mirror (pothoscomms_b200/_abi.py) binds the same symbols for tests and bench.
 *
 * Every entry point cites the reference interface it replaces (paths relative to the
 * PothosComms checkout).  A handle is used by one thread at a time (the Pothos actor model:
 * work() and registered calls of one block never overlap); distinct handles are independent.
 * There is NO CPU fallback: every compute call fails with B200C_ERR_CUDA when no sm_100
 * device is usable.
 */
#ifndef B200COMMS_H
#define B200COMMS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200C_ABI_VERSION 2

/* status codes */
#define B200C_OK 0
#define B200C_ERR_INVALID (-1)     /* Pothos::InvalidArgumentException in the block layer */
#define B200C_ERR_UNSUPPORTED (-2) /* "unsupported types" factory errors */
#define B200C_ERR_CUDA (-3)        /* CUDA runtime / driver failure, or no usable device */
#define B200C_ERR_NOMEM (-4)

/* Element types = the rows of FIRFilterFactory (filter/FIRFilter.cpp:377-382) and FFTFactory
 * (fft/FFT.cpp:89-91).  Odd codes are std::complex<T> stored interleaved (re, im). */
enum b200c_dtype {
    B200C_F32 = 0, B200C_CF32 = 1,
    B200C_F64 = 2, B200C_CF64 = 3,
    B200C_I8 = 4, B200C_CI8 = 5,
    B200C_I16 = 6, B200C_CI16 = 7,
    B200C_I32 = 8, B200C_CI32 = 9,
    B200C_I64 = 10, B200C_CI64 = 11
};

/* tapsType argument of the factory: "REAL" / "COMPLEX" (filter/FIRFilter.cpp:373-376) */
enum b200c_taps_kind { B200C_TAPS_REAL = 0, B200C_TAPS_COMPLEX = 1 };

/* thread-local text of the last error on the calling thread */
const char *b200c_last_error(void);
int b200c_abi_version(void);
/* number of CUDA devices; 0 (and B200C_OK) when the driver is absent */
int b200c_device_count(int *count);
size_t b200c_dtype_size(int dtype);

/* ------------------------------------------- HBM-resident neighbours (SURVEY 8f rank 4) --- */
/* /comms/scale: arrayScale() with setFactor()'s floatToQ, math/Scale.cpp:15-23,41-45; every row
 * of scaleFactory (:147-153).  `elems` elements of `dtype` (a complex element is one element;
 * a vector dimension multiplies elems).  d_in == d_out is allowed. */
int b200c_scale(int dtype, double factor, const void *d_in, void *d_out, size_t elems, int device, void *stream);
/* /comms/rotate: arrayRotate() with setPhase()'s floatToQ(polar(1, phase)), math/Rotate.cpp:15-23,
 * 71-75; complex types only (rotateFactory :145-157), else B200C_ERR_UNSUPPORTED. */
int b200c_rotate(int dtype, double phase, const void *d_in, void *d_out, size_t elems, int device, void *stream);
/* /comms/signal_probe work(), utility/SignalProbe.cpp:140-160 over one window of `elems` elements:
 * mode 0 VALUE (last element), 1 RMS, 2 MEAN; value[0] = re, value[1] = im (0 for real types and
 * RMS).  Synchronous: the result is on the host when the call returns. */
enum b200c_probe_mode { B200C_PROBE_VALUE = 0, B200C_PROBE_RMS = 1, B200C_PROBE_MEAN = 2 };
int b200c_probe(int dtype, int mode, const void *d_in, size_t elems, double *value, int device, void *stream);
/* The work() loops of /comms/waveform_source and /comms/noise_source (fast mode):
 *   out[i] = table[(index + i*step) & (table_elems - 1)],  i < elems
 * waveform/WaveformSource.cpp:98-108 (step = _step, the caller then advances _index by elems*step)
 * and waveform/NoiseSource.cpp:108-117 (step = 1, 4096 entries).  d_table: table_elems elements of
 * `dtype` in DEVICE memory, filled by the block layer as updateTable() does (WaveformSource.cpp:184-260,
 * NoiseSource.cpp:188-226); table_elems must be a power of two (the reference's mask) else
 * B200C_ERR_INVALID.  Every row of the two factories (all twelve types).  Asynchronous on `stream`. */
int b200c_table_source(int dtype, const void *d_table, size_t table_elems, uint64_t index, uint64_t step, void *d_out,
                       size_t elems, int device, void *stream);

/* ------------------------------------------------------------------ /comms/fir_filter --- */
typedef struct b200c_fir b200c_fir;

/* FIRFilterFactory(dtype, tapsType) + FIRFilter::FIRFilter(), filter/FIRFilter.cpp:369-384,
 * 102-126: M = L = 1, taps = {1}.  Real data with COMPLEX taps -> B200C_ERR_UNSUPPORTED. */
int b200c_fir_create(b200c_fir **out, int dtype, int taps_kind, int device);
int b200c_fir_destroy(b200c_fir *h);

/* setTaps(), filter/FIRFilter.cpp:138-144 and updateInternals() :327-354.  `taps` holds ntaps
 * doubles ("REAL") or ntaps (re, im) double pairs ("COMPLEX").  ntaps == 0 -> B200C_ERR_INVALID.
 * Does the per-phase split and floatToQ (:340-350) on the host, then uploads the tap table. */
int b200c_fir_set_taps(b200c_fir *h, const double *taps, size_t ntaps);
/* setDecimation()/setInterpolation(), filter/FIRFilter.cpp:151-168; 0 -> B200C_ERR_INVALID */
int b200c_fir_set_rates(b200c_fir *h, size_t decim, size_t interp);
/* K (:335) and _inputRequire = M + K - 1 (:353) */
int b200c_fir_info(const b200c_fir *h, size_t *K, size_t *input_require, size_t *decim, size_t *interp);
/* Name of the device kernel family b200c_fir_run() launches for the current taps/rates (diagnostic, used by
 * bench.py's roofline record): "fir_os32_kernel" / "fir_os64p_kernel" / "fir_os32r_kernel" / "fir_os32x_kernel" /
 * "fir_ospg_kernel" / "fir_osp_kernel" / "fir_os32g_kernel" (fused fast convolution, float streams),
 * "fir_umma32_kernel" / "fir_umma_kernel" / "fir_ummap_kernel" / "fir_imma_kernel" (int16 on the int8 tensor cores),
 * "fir_tile_kernel" / "fir_generic_kernel" (direct form). */
const char *b200c_fir_kernel(const b200c_fir *h);

/* The N arithmetic of work(), filter/FIRFilter.cpp:278:
 *   N = min((elems - (K-1)) / M, out_capacity / L) * M, elems = in_elems (+ K-1 if zero_tail)
 * consume = N, produce = (N/M)*L (:307-308).  Host only, no device work. */
int b200c_fir_plan(const b200c_fir *h, size_t in_elems, size_t out_capacity, int zero_tail,
                   size_t *consume, size_t *produce);

/* The convolution nest of work(), filter/FIRFilter.cpp:281-302, on DEVICE buffers.
 * d_in: in_elems elements, the first K-1 are history (:281).  zero_tail != 0 treats K-1
 * further elements as zeros (burst flush, :265-272) without materialising them.
 * d_out: room for out_capacity elements.  Stateless in the stream history, asynchronous on
 * `stream` (a cudaStream_t; NULL = default stream).  Writes *consumed / *produced as
 * b200c_fir_plan() would. */
int b200c_fir_run(b200c_fir *h, const void *d_in, size_t in_elems, void *d_out, size_t out_capacity,
                  int zero_tail, size_t *consumed, size_t *produced, void *stream);

/* Same call with HOST buffers (what a host-domain Pothos neighbour hands the block): chunked
 * H2D -> kernel -> D2H, double-buffered over two streams, synchronous on return. */
int b200c_fir_run_host(b200c_fir *h, const void *h_in, size_t in_elems, void *h_out, size_t out_capacity,
                       int zero_tail, size_t *consumed, size_t *produced);

/* ------------------------------------------------------- bank of /comms/fir_filter blocks --- */
/* `nchan` independent FIRFilter instances of one element type (one per channel of a channeliser /
 * filter bank: every reference block instance holds all of its own state, filter/FIRFilter.cpp:356-363),
 * driven together: channel c reads d_in + c*in_stride and writes d_out + c*out_stride (strides in
 * elements), all channels see the same in_elems / out_capacity, so consume / produce are common.
 * Every channel has its own taps (b200c_fir_bank_set_taps) but the same tap COUNT and rates.
 * complex float32 streams at L = M = 1 run as ONE launch over (channel, block); other types and
 * rates run the channels' kernels back to back on `stream`.  Results per channel are b200c_fir_run's. */
typedef struct b200c_fir_bank b200c_fir_bank;
int b200c_fir_bank_create(b200c_fir_bank **out, int dtype, int taps_kind, size_t nchan, int device);
int b200c_fir_bank_destroy(b200c_fir_bank *b);
int b200c_fir_bank_set_taps(b200c_fir_bank *b, size_t chan, const double *taps, size_t ntaps);
int b200c_fir_bank_set_rates(b200c_fir_bank *b, size_t decim, size_t interp);
int b200c_fir_bank_info(const b200c_fir_bank *b, size_t *nchan, size_t *K, size_t *input_require);
int b200c_fir_bank_run(b200c_fir_bank *b, const void *d_in, size_t in_stride, size_t in_elems, void *d_out,
                       size_t out_stride, size_t out_capacity, int zero_tail, size_t *consumed, size_t *produced,
                       void *stream);

/* ------------------------------------- polyphase filter-bank channelizer (one stream in) --- */
/* Splits ONE wideband complex float32 stream into `nchan` = M baseband channels, decimated by `decim` = D.
 * Channel c is exactly /comms/fir_filter with REAL taps h, decimation D (filter/FIRFilter.cpp:278-302: it
 * emits on the last of every D inputs) applied to the stream mixed down by c/M cycles per sample:
 *   z[i] = x[i] exp(-2 pi i c (s + i) / M),     s = stream_index = absolute stream index of d_in[0]
 * i.e., with m_t = (ntaps-1) + t D + (D-1) the newest input sample of output frame t,
 *   y_c[t] = sum_{n < ntaps} h[n] x[m_t - n] exp(-2 pi i c (s + m_t - n) / M).
 * Channel c is centred at +c/M cycles per sample; channels c >= M/2 are the negative frequencies.  Only
 * s mod M matters, so a stream cut into pieces (or segments on several GPUs) keeps its channel phases as long as
 * each call passes the absolute index of its first element.
 * Computed as a polyphase filter bank: ceil(ntaps/M) real-tap products per branch and frame, then one M-point
 * FFT per frame; each input sample is read about once and each output written once.
 *
 * dtype B200C_CF32 only, M a power of two in [2, 4096] (else B200C_ERR_UNSUPPORTED); D >= 1 dividing M (D = M:
 * critically sampled, D = M/2: 2x oversampled) and 1 <= ntaps <= 16 M (else B200C_ERR_INVALID).  Create-time
 * arguments are checked before any device call.  Taps: real doubles stored as float32, {1} after create. */
typedef struct b200c_chan b200c_chan;
int b200c_chan_create(b200c_chan **out, int dtype, size_t nchan, size_t decim, int device);
int b200c_chan_destroy(b200c_chan *h);
int b200c_chan_set_taps(b200c_chan *h, const double *taps, size_t ntaps);
/* input_require = ntaps - 1 + decim */
int b200c_chan_info(const b200c_chan *h, size_t *nchan, size_t *decim, size_t *ntaps, size_t *input_require);
/* d_in: in_elems complex float32 samples on the device, the first ntaps-1 of them history (as b200c_fir_run with
 * K = ntaps, L = 1).  F = min((in_elems - (ntaps-1)) / D, out_capacity), 0 when in_elems < ntaps-1+D;
 * *consumed = F D, *produced = F.  Frame t of channel c goes to d_out[c * out_stride + t] (elements): the layout
 * b200c_fir_bank_run reads, so the channels can be post-filtered by a bank without a copy.  Nothing else of d_out
 * is written.  Null buffers (with F > 0) or out_stride < F -> B200C_ERR_INVALID.  Stateless, asynchronous on
 * `stream`, one kernel launch; a frame's value does not depend on how the stream was cut into calls (bit for bit). */
int b200c_chan_run(b200c_chan *h, const void *d_in, size_t in_elems, uint64_t stream_index, void *d_out, size_t out_stride,
                   size_t out_capacity, size_t *consumed, size_t *produced, void *stream);

/* --------------------------- real-input polyphase filter-bank channelizer (one real stream in) --- */
/* The channelizer above applied to ONE real stream x of float32 or int16 (what direct-IF / direct-RF sampling
 * digitizers deliver), keeping only the channels that are not complex-conjugate mirrors.  With M = branches, D =
 * decim, s = stream_index (the absolute index of d_in[0]) and m_t = (ntaps-1) + t D + (D-1), for c = 0 .. M/2
 *   y_c[t] = sum_{n < ntaps} h[n] x[m_t - n] exp(-2 pi i c (s + m_t - n) / M).
 * Channel c is centred at +c/M cycles per sample; the channels M/2 < c < M of the complex definition are
 * conj(y_{M-c}) and are not produced.  Channels 0 and M/2 are real: their imaginary parts are written as exactly 0.
 * Only s mod M matters.  int16 samples are converted to float32 exactly (no scaling), so int16 input gives output
 * bit-identical to float32 input of the same values.
 * Computed as a polyphase filter bank: ceil(ntaps/M) real products per branch and frame, the real M-point frame
 * packed into one M/2-point complex FFT (within the frame, never two frames together), then the even/odd split.
 *
 * dtype B200C_F32 or B200C_I16 (else B200C_ERR_UNSUPPORTED); M a power of two in [2, 8192] (else
 * B200C_ERR_UNSUPPORTED); D >= 1 dividing M (else B200C_ERR_INVALID).  Checked before any device call.  Taps: real
 * doubles stored as float32, {1} after create; 1 <= ntaps <= 16 M, else B200C_ERR_INVALID and the old taps stay. */
typedef struct b200c_rchan b200c_rchan;
int b200c_rchan_create(b200c_rchan **out, int dtype, size_t m, size_t decim, int device);
int b200c_rchan_destroy(b200c_rchan *h);
int b200c_rchan_set_taps(b200c_rchan *h, const double *taps, size_t ntaps);
/* nchan = M/2 + 1 output rows; input_require = ntaps - 1 + decim */
int b200c_rchan_info(const b200c_rchan *h, size_t *m, size_t *nchan, size_t *decim, size_t *ntaps, size_t *input_require);
/* d_in: in_elems real samples of the handle's dtype on the device, the first ntaps-1 of them history; it may start
 * at any element offset.  F = min((in_elems - (ntaps-1)) / D, out_capacity), 0 when in_elems < ntaps-1+D;
 * *consumed = F D, *produced = F.  Frame t of channel c (c <= M/2) goes to d_out[c * out_stride + t] (complex
 * float32 elements): the layout b200c_fir_bank_run reads, so a complex float32 bank of M/2 + 1 channels can
 * post-filter them without a copy.  Nothing else of d_out is written.  Null buffers (with F > 0) or out_stride < F
 * -> B200C_ERR_INVALID.  Stateless, asynchronous on `stream`, one kernel launch; a frame's value does not depend on
 * how the stream was cut into calls (bit for bit). */
int b200c_rchan_run(b200c_rchan *h, const void *d_in, size_t in_elems, uint64_t stream_index, void *d_out,
                    size_t out_stride, size_t out_capacity, size_t *consumed, size_t *produced, void *stream);

/* --------------------------------- polyphase synthesis filter bank (one stream out) --- */
/* The transpose of the channelizer: puts `nchan` = M baseband channels, interpolated by `interp` = D, back into
 * ONE wideband complex float32 stream.  Channel c goes through /comms/fir_filter with REAL taps g, interpolation
 * D and decimation 1, is mixed up by +c/M cycles per sample, and all channels are summed.  With K = ceil(ntaps/D)
 * and s = stream_index, the absolute stream index of d_out[0], output sample m = t D + j (j < D) is
 *   y[t D + j] = sum_{c < M} exp(+2 pi i c (s + t D + j) / M) sum_{k < K, j + k D < ntaps} g[j + k D] X_c[K-1 + t - k]
 * Channels c >= M/2 are the negative frequencies (the channelizer's convention).  Only s mod M matters.
 * Computed as a polyphase synthesizer: one inverse M-point FFT per input frame, then K real-tap products per
 * output sample; each input frame is read about once and each output sample written once.
 *
 * dtype B200C_CF32 only, M a power of two in [2, 4096] (else B200C_ERR_UNSUPPORTED); D >= 1 dividing M (D = M:
 * critically sampled, D = M/2: 2x oversampled) and 1 <= ntaps <= min(16 M, 32 D), so K <= 32 (else
 * B200C_ERR_INVALID; a refused set_taps keeps the old taps).  Create-time arguments are checked before any device
 * call.  Taps: real doubles stored as float32, {1} after create.
 *
 * Perfect reconstruction after b200c_chan with D = M/2 (INTEGRATION §1): analysis h = firwin(12M+1, 1/M,
 * kaiser 10), synthesis g = D firwin(28D+1, 2/M, kaiser_beta(90)); synthesizer stream_index
 * s_a + (ntaps_h - 1) + (D - 1) + (K_g - 1) D, where s_a is the channelizer's. */
typedef struct b200c_synth b200c_synth;
int b200c_synth_create(b200c_synth **out, int dtype, size_t nchan, size_t interp, int device);
int b200c_synth_destroy(b200c_synth *h);
int b200c_synth_set_taps(b200c_synth *h, const double *taps, size_t ntaps);
/* input_require = K frames per channel */
int b200c_synth_info(const b200c_synth *h, size_t *nchan, size_t *interp, size_t *ntaps, size_t *input_require);
/* d_in: M channel rows in the channelizer's output layout, frame i of channel c at d_in[c * in_stride + i] for
 * i < in_frames; the first K-1 frames of every channel are history (as b200c_fir_run with L = D, M = 1).
 * F = min(in_frames - (K-1), out_capacity / D), 0 when in_frames < K; *consumed = F frames per channel,
 * *produced = F D samples, written to d_out[0 .. F D) and nowhere else.  Null buffers (with F > 0) or
 * in_stride < in_frames -> B200C_ERR_INVALID.  Stateless, asynchronous on `stream`, one kernel launch; an output
 * sample's value does not depend on how the stream was cut into calls (bit for bit). */
int b200c_synth_run(b200c_synth *h, const void *d_in, size_t in_stride, size_t in_frames, uint64_t stream_index, void *d_out,
                    size_t out_capacity, size_t *consumed, size_t *produced, void *stream);

/* ------------------------- real-output polyphase synthesis filter bank (one real stream out) --- */
/* The transpose of the real-input channelizer: puts the M/2 + 1 rows c = 0 .. M/2 that b200c_rchan_run writes back
 * into ONE real stream of float32 or int16 (what direct-IF / direct-RF DACs take).  With M = branches, N = M/2,
 * D = interp, K = ceil(ntaps/D) and s = stream_index, the absolute stream index of d_out[0], output sample
 * m = t D + j (j < D) is
 *   y[t D + j] = sum_{k < K} g[j + k D] sum_{c = 0..N} w_c Re( exp(+2 pi i c (s + t D + j) / M) X_c[K-1 + t - k] ),
 *   w_0 = w_N = 1, w_c = 2 otherwise   (g zero beyond ntaps),
 * i.e. the real part of b200c_synth_run's output at M channels when rows M - c are conj(X_c) for 0 < c < N.  Only
 * the real parts of rows 0 and N are read.  Only s mod M matters.  int16 output is the float32 result rounded to
 * nearest (ties to even) and saturated to [-32768, 32767], with no other scaling: bit-identical to clamping and
 * rounding the float32 output of the same taps and input.  Non-finite values give unspecified int16 samples.
 * Computed as a polyphase synthesizer: the real inverse M-point DFT of each input frame packed into one M/2-point
 * complex inverse FFT (within the frame, never two frames together), then K real-tap products per output sample.
 *
 * dtype (the output) B200C_F32 or B200C_I16 (else B200C_ERR_UNSUPPORTED); M a power of two in [2, 8192] (else
 * B200C_ERR_UNSUPPORTED); D >= 1 dividing M (else B200C_ERR_INVALID).  Checked before any device call.  Taps: real
 * doubles stored as float32, {1} after create; 1 <= ntaps <= min(16 M, 32 D), else B200C_ERR_INVALID and the old
 * taps stay.
 *
 * Perfect reconstruction after b200c_rchan with D = M/2: the complex pair's recipe (b200c_synth above) unchanged. */
typedef struct b200c_rsynth b200c_rsynth;
int b200c_rsynth_create(b200c_rsynth **out, int dtype, size_t m, size_t interp, int device);
int b200c_rsynth_destroy(b200c_rsynth *h);
int b200c_rsynth_set_taps(b200c_rsynth *h, const double *taps, size_t ntaps);
/* nchan = M/2 + 1 input rows; input_require = K frames per row */
int b200c_rsynth_info(const b200c_rsynth *h, size_t *m, size_t *nchan, size_t *interp, size_t *ntaps, size_t *input_require);
/* d_in: M/2 + 1 rows of complex float32 in the real channelizer's output layout, frame i of row c at
 * d_in[c * in_stride + i] for i < in_frames; the first K-1 frames of every row are history.
 * F = min(in_frames - (K-1), out_capacity / D), 0 when in_frames < K; *consumed = F frames per row, *produced = F D
 * samples of the handle's dtype, written to d_out[0 .. F D) and nowhere else; d_out may start at any element offset.
 * Null buffers (with F > 0) or in_stride < in_frames -> B200C_ERR_INVALID.  Stateless, asynchronous on `stream`,
 * one kernel launch; an output sample's value does not depend on how the stream was cut into calls (bit for bit). */
int b200c_rsynth_run(b200c_rsynth *h, const void *d_in, size_t in_stride, size_t in_frames, uint64_t stream_index,
                     void *d_out, size_t out_capacity, size_t *consumed, size_t *produced, void *stream);

/* ------------------------------------------------------------------------- /comms/fft --- */
typedef struct b200c_fft b200c_fft;

/* FFTFactory(dtype, numBins, inverse) + FFTAux, fft/FFT.cpp:83-93, fft/FFTAux.h:16-48.
 * dtype in {CF32, CF64, CI16}; anything else -> B200C_ERR_UNSUPPORTED (fft/FFT.cpp:92).
 * Float types: unnormalised both ways (fft/kissfft.hh); CI16: Q15 kiss_fft, 1/N both ways. */
int b200c_fft_create(b200c_fft **out, int dtype, size_t nbins, int inverse, int device);
int b200c_fft_destroy(b200c_fft *h);
int b200c_fft_info(const b200c_fft *h, size_t *nbins, int *inverse);
/* `batch` back-to-back transforms == `batch` work() calls of fft/FFT.cpp:61-72 (each consumes
 * and produces nbins elements).  Device buffers, asynchronous on `stream`. */
int b200c_fft_run(b200c_fft *h, const void *d_in, void *d_out, size_t batch, void *stream);
int b200c_fft_run_host(b200c_fft *h, const void *h_in, void *h_out, size_t batch);

/* ----------------------------------------------- device-resident buffers (BufferManager) --- */
/* Backing store of the block layer's device BufferManagers, replacing
 * Pothos::BufferManager::make("circular") (filter/FIRFilter.cpp:196-199) and
 * make("generic", args) (fft/FFT.cpp:54-59).  A ring is `bytes` of HBM mapped twice back to
 * back in virtual address space (CUDA VMM), so [base + off, base + off + len) is contiguous
 * for any off < bytes, len <= bytes: the K-1 history samples always sit contiguously in
 * front of new data with zero copies. */
typedef struct b200c_ring b200c_ring;
int b200c_ring_create(b200c_ring **out, size_t min_bytes, int device);
int b200c_ring_destroy(b200c_ring *r);
void *b200c_ring_base(const b200c_ring *r);
size_t b200c_ring_bytes(const b200c_ring *r);

int b200c_dev_alloc(void **d_ptr, size_t bytes, int device);
int b200c_dev_free(void *d_ptr, int device);
int b200c_host_alloc_pinned(void **h_ptr, size_t bytes);
int b200c_host_free_pinned(void *h_ptr);
int b200c_copy_h2d(void *d_dst, const void *h_src, size_t bytes, int device, void *stream);
int b200c_copy_d2h(void *h_dst, const void *d_src, size_t bytes, int device, void *stream);
int b200c_copy_d2d(void *d_dst, const void *d_src, size_t bytes, int device, void *stream);
int b200c_memset(void *d_dst, int value, size_t bytes, int device, void *stream);
int b200c_stream_sync(int device, void *stream);

/* ------------------------------------------- multi-GPU: the K-1 halo (SURVEY.md 8e) --- */
/* One long stream cut into contiguous segments, one per GPU, every segment start a multiple of M (the
 * decimation counter restarts at M in every work() call, filter/FIRFilter.cpp:283,291-292).  The only
 * dependency between segments is the K-1 samples of left history (:281,298): GPU r keeps its segment as
 * [K-1 halo | n samples] and, before each pass, pulls the last K-1 samples of GPU r-1's segment into the
 * halo -- b200c_halo_exchange, ONE copy over NVLink enqueued on the consumer's compute stream.  GPU 0's
 * halo is the stream's true first K-1 samples (history only, as in the reference).  No torch, no
 * collective library: a C++ Pothos host shards a stream with these calls alone.
 *
 * One process per GPU: the owner exports a range of device memory (cudaMalloc-backed: b200c_dev_alloc or
 * a framework allocator's block) as a plain 128-byte record, the host program carries the record to the
 * neighbour process however it likes, the neighbour opens it.  When exporter and opener are the same
 * process the pointer is used directly (peer access is enabled on first use). */
typedef struct b200c_peer_mem {
    unsigned char ipc[64];   /* cudaIpcMemHandle_t of the allocation that holds the range */
    uint64_t offset, bytes;  /* the range inside it */
    uint64_t local_ptr;      /* the exporter's own pointer (meaningful in the exporting process only) */
    int64_t pid;             /* exporting process */
    int32_t device;          /* exporter's device ordinal */
    int32_t reserved[7];
} b200c_peer_mem;
int b200c_peer_export(const void *d_ptr, size_t bytes, int device, b200c_peer_mem *out);
/* *d_peer_ptr: the range, addressable from `device`; *mapping: token for b200c_peer_close */
int b200c_peer_open(const b200c_peer_mem *m, int device, void **d_peer_ptr, void **mapping);
int b200c_peer_close(void *mapping);

/* Ordering between the producer of a segment's tail and the neighbour that pulls it: an interprocess
 * event.  The owner records it on its stream once the tail is final; the neighbour makes its compute
 * stream wait for it before b200c_halo_exchange. */
typedef struct b200c_peer_event {
    unsigned char ipc[64];   /* cudaIpcEventHandle_t */
    uint64_t local_event;    /* meaningful in the creating process only */
    int64_t pid;
    int32_t reserved[12];
} b200c_peer_event;
int b200c_peer_event_create(void **event, int device, b200c_peer_event *out);
int b200c_peer_event_open(const b200c_peer_event *e, int device, void **event);
int b200c_peer_event_record(void *event, int device, void *stream);
int b200c_peer_event_wait(void *event, int device, void *stream);
int b200c_peer_event_destroy(void *event, int device);

/* d_halo_dst[0 .. bytes) = d_peer_tail[0 .. bytes), bytes = (K-1) * element size, asynchronous on `stream`
 * (the stream b200c_fir_run is then given).  d_peer_tail comes from b200c_peer_open. */
int b200c_halo_exchange(void *d_halo_dst, const void *d_peer_tail, size_t bytes, int device, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* B200COMMS_H */
