/* qpskcuda.h — C ABI of libqpskcuda.so, the B200 (sm_100a) hot path behind the C# QPSK modem
 * NustyFrozen/QPSK-Modulator-Demodulator.
 *
 * The reference has no FFI of its own: the boundary is its public C# class surface
 * (SURVEY.md §8b).  Every entry point below names the reference member it stands in for
 * ("MS/" = Modulation-Simulation/, "TB/" = TestBench/).  INTEGRATION.md shows the
 * [DllImport("qpskcuda")] stubs a maintainer adds to those classes.
 *
 * Conventions
 *   - samples are interleaved float IQ ([I0,Q0,I1,Q1,...]) exactly like the C# spans; lengths
 *     named n_floats count floats (2 per complex sample), like Span<float>.Length.
 *   - every function returns a status (0 ok, <0 error).  The negative codes map 1:1 onto the
 *     exceptions the reference throws at the same place.
 *   - handles are opaque, own their device state and CUDA streams, and are not thread-safe
 *     (the reference objects are not either); different handles may be used concurrently.
 *   - "host" entry points take host pointers and copy through the device inside the call;
 *     "_dev" entry points take device pointers (16-byte aligned) and enqueue on `stream`
 *     (a cudaStream_t passed as void*; NULL = the handle's own stream) without synchronising.
 *   - there is no CPU fallback: without a CUDA device every compute call returns
 *     QPSK_ERR_NO_DEVICE / QPSK_ERR_CUDA.
 */
#ifndef QPSKCUDA_H_
#define QPSKCUDA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define QPSK_API __declspec(dllexport)
#else
#define QPSK_API __attribute__((visibility("default")))
#endif

/* ---- status codes ------------------------------------------------------------------------ */
#define QPSK_OK 0
#define QPSK_ERR_NULL (-1)        /* ArgumentNullException                                       */
#define QPSK_ERR_ARG (-2)         /* ArgumentException (odd IQ length, empty taps, short output) */
#define QPSK_ERR_RANGE (-3)       /* ArgumentOutOfRangeException (bad design parameter)          */
#define QPSK_ERR_CUDA (-4)        /* a CUDA runtime call failed; see qpsk_last_cuda_error()      */
#define QPSK_ERR_NOMEM (-5)       /* host or device allocation failed                            */
#define QPSK_ERR_CAPACITY (-6)    /* caller buffer too small; the needed size is reported        */
#define QPSK_ERR_UNSUPPORTED (-7) /* outside the limits stated in DESIGN.md                      */
#define QPSK_ERR_NO_DEVICE (-8)   /* no CUDA device / wrong architecture                         */

typedef struct qpsk_fir qpsk_fir;
typedef struct qpsk_fll qpsk_fll;
typedef struct qpsk_mm qpsk_mm;
typedef struct qpsk_costas qpsk_costas;
typedef struct qpsk_mod qpsk_mod;
typedef struct qpsk_demod qpsk_demod;
typedef struct qpsk_chan qpsk_chan;
typedef struct qpsk_chain qpsk_chain;
typedef struct qpsk_stream qpsk_stream;

/* ---- library / device -------------------------------------------------------------------- */
QPSK_API int qpsk_version(void);                       /* 10000*major + 100*minor + patch         */
/* build stamp: hash of the kernel sources, this header, the nvcc flags and version the library was compiled from (16 hex
 * chars).  The Python host refuses a library whose stamp differs from the source tree next to it; bench.py prints it. */
QPSK_API const char* qpsk_build_id(void);
QPSK_API const char* qpsk_strerror(int status);
QPSK_API const char* qpsk_last_cuda_error(void);       /* thread-local text of the last CUDA error */
QPSK_API int qpsk_device_count(int* n);
QPSK_API int qpsk_set_device(int ordinal);             /* device used by handles created afterwards */
QPSK_API int qpsk_device_info(int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes);
/* pinned host memory so host entry points overlap PCIe copies with kernels (optional) */
QPSK_API int qpsk_host_alloc(void** p, int64_t bytes);
QPSK_API int qpsk_host_free(void* p);
/* page-lock / unlock caller-owned memory in place (e.g. a C# float[] held by a pinned GCHandle): a GC pin keeps
 * the array from moving but leaves it pageable, and pageable copies are staged by the driver at a fraction of the
 * PCIe rate.  Registering once per long-lived buffer gives the host entry points the same copy rate as
 * qpsk_host_alloc memory. */
QPSK_API int qpsk_host_register(void* p, int64_t bytes);
QPSK_API int qpsk_host_unregister(void* p);
/* launches of this library's kernels issued by the calling thread since the last reset */
QPSK_API int64_t qpsk_launch_count(void);
QPSK_API void qpsk_launch_count_reset(void);

/* ---- a1  RRCFilter.generateCoefficents  (MS/Models/RRC-filter.cs:16-75) ------------------- */
/* host-side fp64 design.  out==NULL or cap too small: *n is still set (size query). */
QPSK_API int qpsk_rrc_taps(double span_symbols, double beta, int sample_rate, int symbol_rate,
                           double* out, int cap, int* n);

/* ---- a2-a5  ComplexFIRFilter  (MS/Models/FIRFilter.cs:8-232) ------------------------------ */
#define QPSK_FIR_FAST 0   /* fp32 FMA accumulation (default); the library picks the kernel: for real taps from
                           * 47 taps on the 2-parallel split below, else the tap-sequential FMA kernel          */
#define QPSK_FIR_EXACT 1  /* the reference's summation order: 8 lane partials, no FMA (:165-192) */
#define QPSK_FIR_FMA 2    /* always the tap-sequential FMA kernel (one rounding per tap)                         */
#define QPSK_FIR_SPLIT 3  /* the 2-parallel fast-FIR split wherever it applies (real taps, >= 14 taps): three half-length
                           * sub-filters per output pair, 0.8 of the multiply-adds; other summation order, still within
                           * 1e-5 of max|y| of the reference.  Outputs are NOT bit-identical across different chunkings
                           * of one stream (a cancelled term contains the following sample); FMA and EXACT are.    */
/* ctor :29-53.  taps_iq interleaved complex taps; n_floats even and > 0. */
QPSK_API int qpsk_fir_create(const float* taps_iq, int n_floats, qpsk_fir** out);
/* the same filter over `channels` independent streams, one (N-1)-sample history each */
QPSK_API int qpsk_fir_create_batch(const float* taps_iq, int n_floats, int channels, qpsk_fir** out);
QPSK_API int qpsk_fir_destroy(qpsk_fir* f);
QPSK_API int qpsk_fir_reset(qpsk_fir* f);                      /* zero the delay line(s)          */
QPSK_API int qpsk_fir_set_mode(qpsk_fir* f, int mode);
QPSK_API int qpsk_fir_num_taps(const qpsk_fir* f, int* n_complex);
/* name of the kernel the handle's last filter call launched (which of the kernels in DESIGN.md §3 served it) */
QPSK_API int qpsk_fir_last_kernel(const qpsk_fir* f, char* name, int cap);
/* Filter(ReadOnlySpan<float>, Span<float>) :80-91 — streaming, same length, history kept.
 * out_cap_floats < n_floats -> QPSK_ERR_ARG (:83); odd n_floats -> QPSK_ERR_ARG (:82).
 * Batch handles: in/out are [channels][n_floats] contiguous. */
QPSK_API int qpsk_fir_filter(qpsk_fir* f, const float* iq_in, float* iq_out, int64_t n_floats,
                             int64_t out_cap_floats);
/* fftFilter(float[]) :96-141 — stateless, y[i] = conv(x,h)[i + N-1], i < n. */
QPSK_API int qpsk_fir_fft_filter(qpsk_fir* f, const float* iq_in, float* iq_out, int64_t n_floats);
/* device-resident variants; strides are in floats between consecutive channels */
QPSK_API int qpsk_fir_filter_dev(qpsk_fir* f, const float* d_in, float* d_out, int64_t n_floats,
                                 int64_t in_stride_floats, int64_t out_stride_floats, void* stream);
QPSK_API int qpsk_fir_fft_filter_dev(qpsk_fir* f, const float* d_in, float* d_out, int64_t n_floats,
                                     int64_t in_stride_floats, int64_t out_stride_floats, void* stream);
/* Decimate-by-D matched filter (north_star item (2); SURVEY §8d "decimate-by-D variant").  The reference's matched filter is
 * non-decimating (FIRFilter.cs:80-91, called at QPSKDeModulator.cs:360), so this is defined by it: the streaming Filter()
 * output kept at indices 0, D, 2D, ... of the samples passed to this call since the handle's creation, its last reset or a
 * change of D — counted ACROSS calls, so any chunking gives the same decimated stream: y_dec[m] = y[m*D].  Only the kept outputs are computed: 4N/D flop (real taps) and
 * 8 + 8/D bytes per input sample.  Shares the delay line with qpsk_fir_filter (the calls may be mixed).  Each channel
 * gets ceil((n - skip)/D) outputs; *n_out_floats = floats written per channel.  out_cap too small -> QPSK_ERR_CAPACITY
 * with no state consumed.  D = 2, 4, 8, 16 with real taps in a FAST mode run fir_dec2_kernel (D = 2, 16-byte aligned rows) / fir_decim_kernel; every other case
 * (QPSK_FIR_EXACT: bit-identical to the subsampled exact filter) filters at full rate and keeps every D-th sample. */
QPSK_API int qpsk_fir_decimate(qpsk_fir* f, const float* iq_in, int64_t n_floats, int decim, float* iq_out,
                               int64_t out_cap_floats, int64_t* n_out_floats);
QPSK_API int qpsk_fir_decimate_dev(qpsk_fir* f, const float* d_in, int64_t n_floats, int64_t in_stride_floats, int decim,
                                   float* d_out, int64_t out_cap_floats, int64_t out_stride_floats, int64_t* n_out_floats,
                                   void* stream);
/* delay-line checkpoint: the last N-1 inputs per channel, oldest first, [channels][2*(N-1)] */
QPSK_API int qpsk_fir_get_state(qpsk_fir* f, float* hist_iq, int64_t cap_floats);
QPSK_API int qpsk_fir_set_state(qpsk_fir* f, const float* hist_iq, int64_t n_floats);

/* ---- a7-a8  FLLBandEdgeFilter  (MS/Models/Band-Edge Filter.cs:14-203) ---------------------- */
/* DesignFilter :132-183, host-side fp32.  lower/upper: 2*filter_size floats each. */
QPSK_API int qpsk_fll_design(float sps, float rolloff, int filter_size, float* lower_iq, float* upper_iq);
QPSK_API int qpsk_fll_create(float sps, float rolloff, int filter_size, float bandwidth, qpsk_fll** out);
QPSK_API int qpsk_fll_create_batch(float sps, float rolloff, int filter_size, float bandwidth,
                                   int channels, qpsk_fll** out);
QPSK_API int qpsk_fll_destroy(qpsk_fll* f);
/* Process(ReadOnlySpan<float>, Span<float>) :64-87 */
QPSK_API int qpsk_fll_process(qpsk_fll* f, const float* iq_in, float* iq_out, int64_t n_floats,
                              int64_t out_cap_floats);
QPSK_API int qpsk_fll_process_dev(qpsk_fll* f, const float* d_in, float* d_out, int64_t n_floats,
                                  int64_t in_stride_floats, int64_t out_stride_floats, void* stream);
/* public fields phase/freq :25-26, per channel */
QPSK_API int qpsk_fll_get_state(qpsk_fll* f, float* phase, float* freq);
QPSK_API int qpsk_fll_set_state(qpsk_fll* f, const float* phase, const float* freq);

/* ---- a9  MuellerMuller  (MS/Models/MuellerMuller.cs:17-250) -------------------------------- */
QPSK_API int qpsk_mm_create(double samples_per_symbol, double kp, double ki, qpsk_mm** out);
QPSK_API int qpsk_mm_create_batch(double samples_per_symbol, double kp, double ki, int channels, qpsk_mm** out);
QPSK_API int qpsk_mm_destroy(qpsk_mm* m);
/* Process(ReadOnlySpan<float>, Span<float>) :52-136.  n_sym: symbols written (per channel for
 * batch handles: n_sym[channels], out is [channels][cap_floats]). */
QPSK_API int qpsk_mm_process(qpsk_mm* m, const float* mf_iq_in, int64_t n_floats, float* sym_iq_out,
                             int64_t cap_floats, int* n_sym);
QPSK_API int qpsk_mm_process_dev(qpsk_mm* m, const float* d_in, int64_t n_floats, int64_t in_stride_floats,
                                 float* d_out, int64_t cap_floats, int64_t out_stride_floats,
                                 int* d_n_sym, void* stream);
/* per channel: baseIndex, mu, ncoIntegral, queued complex samples */
QPSK_API int qpsk_mm_get_state(qpsk_mm* m, int* base_index, double* mu, double* integral, int* queued);
/* setupSymbolSync gains (MS/QPSKDeModulator.cs:39-55) */
QPSK_API int qpsk_mm_gains_from_bw(double symbol_sync_bw, double* kp, double* ki);

/* ---- a10  CostasLoopQpsk  (MS/Models/CostasLoopQpsk.cs:19-131) ------------------------------ */
QPSK_API int qpsk_costas_create(double sample_rate, double loop_bw_hz, double damping, qpsk_costas** out);
QPSK_API int qpsk_costas_create_batch(double sample_rate, double loop_bw_hz, double damping, int channels,
                                      qpsk_costas** out);
QPSK_API int qpsk_costas_destroy(qpsk_costas* c);
/* Process(ReadOnlySpan<float>, Span<float>) :98-114 */
QPSK_API int qpsk_costas_process(qpsk_costas* c, const float* iq_in, float* iq_out, int64_t n_floats,
                                 int64_t out_cap_floats);
/* batch/device: n_sym[channels] valid complex samples per channel (NULL = n_floats/2 for all) */
QPSK_API int qpsk_costas_process_dev(qpsk_costas* c, const float* d_in, float* d_out, int64_t n_floats,
                                     int64_t in_stride_floats, int64_t out_stride_floats,
                                     const int* d_n_sym, void* stream);
/* GetState() :130, per channel */
QPSK_API int qpsk_costas_get_state(qpsk_costas* c, double* theta, double* freq);

/* ---- symbol-spaced blind CMA equalizer ---------------------------------------------------------------- */
/* Not in the reference (its receive chain has no equalizer); the block a GNU Radio PSK receiver puts between clock
 * recovery and the Costas loop, for multipath channels.  One output per input symbol, group delay D = (n_taps-1)/2.
 * fp32, every product and sum rounded separately (no FMA).  State per channel: taps w[0..N-1] (at creation and reset
 * w[D] = 1+0j, the others 0) and the last N-1 inputs (zero before the stream starts).  For each input x_n, with
 * v_k = x_{n-k} (k = 0..N-1):
 *   P_k = w_k * v_k                        re = w.re*v.re - w.im*v.im, im = w.re*v.im + w.im*v.re
 *   s_l = +0.0f, then s_l = s_l + P_k      for k = l (mod 8), k increasing (l = 0..7, re and im separately)
 *   y   = ((s_0 + s_1) + (s_2 + s_3)) + ((s_4 + s_5) + (s_6 + s_7))
 *   d   = (y.re*y.re + y.im*y.im) - modulus
 *   e   = (fminf(fmaxf(y.re*d, -1), 1), fminf(fmaxf(y.im*d, -1), 1))
 *   g_k = e * conj(v_k)                    re = e.re*v.re + e.im*v.im, im = e.im*v.re - e.re*v.im
 *   w_k = w_k - mu*g_k                     (re and im separately, every k, after y is formed);  output y
 * Fractionally spaced form (qpsk_eq_create_fractional): update stride S >= 1, the samples per symbol of a T/S-spaced
 * input.  Each channel also keeps a stream sample counter n (0 at creation and reset).  Every input sample shifts the
 * window, forms y and outputs it as above; d, e, g and the tap update run only when n % S == 0; then n = n + 1.
 * S = 1 is the symbol-spaced equalizer: one update per input.
 * State persists across calls: any chunking of a stream gives the same outputs bit for bit.
 * n_taps 1..64 (else QPSK_ERR_UNSUPPORTED); mu finite and >= 0, modulus finite and > 0 (else QPSK_ERR_RANGE).  modulus
 * 1.0 is |symbol|^2 at this modem's matched-filter output for unit channel gain.  A refused call consumes no state. */
typedef struct qpsk_eq qpsk_eq;
QPSK_API int qpsk_eq_create(int n_taps, float mu, float modulus, qpsk_eq** out);
QPSK_API int qpsk_eq_create_batch(int n_taps, float mu, float modulus, int channels, qpsk_eq** out);
/* T/sps-spaced (fractionally spaced) equalizer: taps update on every sps-th input sample (update stride S = sps above).
 * One output per input sample, group delay (n_taps-1)/2 samples.  sps 1..8 (else QPSK_ERR_UNSUPPORTED); sps 1 is
 * qpsk_eq_create_batch.  Every other qpsk_eq_* entry point works on the handle unchanged. */
QPSK_API int qpsk_eq_create_fractional(int n_taps, float mu, float modulus, int sps, int channels, qpsk_eq** out);
QPSK_API int qpsk_eq_destroy(qpsk_eq* eq);
QPSK_API int qpsk_eq_reset(qpsk_eq* eq);                      /* taps to the centre spike, window and sample counter zeroed */
/* host memory, iq_in / iq_out [channels][n_floats]; odd n_floats -> QPSK_ERR_ARG, out_cap_floats < n_floats -> QPSK_ERR_CAPACITY */
QPSK_API int qpsk_eq_process(qpsk_eq* eq, const float* iq_in, float* iq_out, int64_t n_floats, int64_t out_cap_floats);
/* device memory, strides in floats; d_n_sym[channels] valid complex symbols per channel (NULL = n_floats/2 for all) */
QPSK_API int qpsk_eq_process_dev(qpsk_eq* eq, const float* d_in, float* d_out, int64_t n_floats, int64_t in_stride_floats,
                                 int64_t out_stride_floats, const int* d_n_sym, void* stream);
/* taps [channels][2*n_taps] interleaved IQ; get: cap_floats < channels*2*n_taps -> QPSK_ERR_CAPACITY; set: n_floats must be
 * exactly channels*2*n_taps (else QPSK_ERR_ARG), every value finite (else QPSK_ERR_RANGE) */
QPSK_API int qpsk_eq_get_taps(qpsk_eq* eq, float* taps_iq, int64_t cap_floats);
QPSK_API int qpsk_eq_set_taps(qpsk_eq* eq, const float* taps_iq, int64_t n_floats);

/* ---- a6  QPSKModulator  (MS/QPSKModulator.cs:18-168) ---------------------------------------- */
/* tsc_bits: '0'/'1' string or NULL (null/whitespace = no TSC, :27) */
QPSK_API int qpsk_mod_create(int sample_rate, int symbol_rate, double rrc_alpha, int rrc_span,
                             int differential, const char* tsc_bits, qpsk_mod** out);
QPSK_API int qpsk_mod_destroy(qpsk_mod* m);
QPSK_API int qpsk_mod_taps(const qpsk_mod* m, double* out, int cap, int* n);       /* getCoeef() :32 */
/* Modulate(string,bool) :104-167.  out==NULL: size query (*n_floats set). */
QPSK_API int qpsk_mod_modulate_bits(qpsk_mod* m, const char* bits, int64_t n_bits, int pulse_shaping,
                                    float* iq_out, int64_t cap_floats, int64_t* n_floats);
/* ModulateBytes :54-72 (ModulateTextUtf8 :74-89 = this over UTF-8 bytes) */
/* §8f-4: the same call with the bit string packed MSB-first (what BitPacker.BytesToBitString,
 * MS/Models/HelperFunctions.cs:14-29, expands to one char per bit); identical samples */
QPSK_API int qpsk_mod_modulate_packed(qpsk_mod* m, const uint8_t* packed_bits, int64_t n_bits, int pulse_shaping,
                                      float* iq_out, int64_t cap_floats, int64_t* n_floats);
QPSK_API int qpsk_mod_modulate_bytes(qpsk_mod* m, const uint8_t* payload, int64_t n_payload,
                                     const uint8_t* start_marker, int64_t n_start,
                                     const uint8_t* end_marker, int64_t n_end, int pulse_shaping,
                                     float* iq_out, int64_t cap_floats, int64_t* n_floats);
/* batch, host memory: ModulateBytes :54-72 over `frames` payloads ([frames][n_payload]) -> [frames][out_stride_floats]
 * samples, frames in groups through a 3-slot kernel / copy-out pipeline (the call is bound by the device-to-host copy:
 * 32*sps output bytes per payload byte).  iq_out == NULL: size query. */
QPSK_API int qpsk_mod_modulate_frames(qpsk_mod* m, const uint8_t* payloads, int64_t n_payload, int frames,
                                      const uint8_t* start_marker, int64_t n_start, const uint8_t* end_marker, int64_t n_end,
                                      float* iq_out, int64_t out_stride_floats, int64_t* frame_floats);
/* batch, device-resident: `frames` payloads of n_payload bytes each ([frames][n_payload], device),
 * each framed START|payload|END (+TSC), differential reference reset per frame (:126); writes
 * [frames][frame_floats] to d_iq_out.  *frame_floats is set even when d_iq_out==NULL. */
QPSK_API int qpsk_mod_modulate_frames_dev(qpsk_mod* m, const uint8_t* d_payloads, int64_t n_payload, int frames,
                                          const uint8_t* start_marker, int64_t n_start,
                                          const uint8_t* end_marker, int64_t n_end,
                                          float* d_iq_out, int64_t out_stride_floats, int64_t* frame_floats,
                                          void* stream);

/* ---- a11-a12  QPSKDeModulator  (MS/QPSKDeModulator.cs:11-456) ------------------------------- */
/* use_fll: 0 = as shipped (fll.Process commented out, :359/:435); 1 = run the FLL in front.
 * max_frame_bytes: bound of the framer ring (the reference allocates 300 MB, :58); 0 = 1 MiB. */
QPSK_API int qpsk_demod_create(int sample_rate, int symbol_rate, float rrc_alpha, int rrc_span,
                               double symbol_sync_bw, double costas_loop_bw, double cfo_loop_bw,
                               int differential, const char* tsc_bits, int use_fll,
                               int64_t max_frame_bytes, qpsk_demod** out);
QPSK_API int qpsk_demod_create_batch(int sample_rate, int symbol_rate, float rrc_alpha, int rrc_span,
                                     double symbol_sync_bw, double costas_loop_bw, double cfo_loop_bw,
                                     int differential, const char* tsc_bits, int use_fll,
                                     int64_t max_frame_bytes, int channels, qpsk_demod** out);
QPSK_API int qpsk_demod_destroy(qpsk_demod* d);
/* matched-filter arithmetic.  Default QPSK_FIR_EXACT: bits, frames and payloads are then those of the reference's
 * summation order bit for bit.  QPSK_FIR_FAST accumulates with FMA (outputs within ~1e-7 relative): a decision can differ
 * only where a decision variable lies that close to zero (bench.py counts such channels on its own bursts). */
QPSK_API int qpsk_demod_set_fir_mode(qpsk_demod* d, int mode);
/* Opt-in CMA equalizer stage (qpsk_eq_* above) between Mueller-Muller and Costas, for multipath channels; n_taps 0 = off
 * (the default: the chain is then exactly the reference's).  The first (n_taps-1)/2 equalizer outputs of each channel's
 * stream are discarded once, so the k-th symbol reaching Costas is the equalized k-th Mueller-Muller symbol (bit
 * alignment as without the stage); the last (n_taps-1)/2 symbols of a call come out at the start of the next.  May be
 * called at any time: synchronises the handle, resets the equalizer (taps, window, discard count) and leaves every other
 * piece of loop and framer state alone.  With the stage on, the symbol path runs as separate MM / EQ / decode kernels. */
QPSK_API int qpsk_demod_set_equalizer(qpsk_demod* d, int n_taps, float mu, float modulus);
/* the equalizer taps, [channels][2*n_taps]; QPSK_ERR_ARG when the stage is off */
QPSK_API int qpsk_demod_equalizer_taps(qpsk_demod* d, float* taps_iq, int64_t cap_floats);
/* Opt-in fractionally spaced CMA equalizer stage (qpsk_eq_create_fractional, S = fs/rs) between the matched filter and
 * Mueller-Muller, so clock recovery locks on an equalized eye; n_taps 0 = off (the default).  Needs an integer rate:
 * fs % rs == 0 and S in 2..8, else QPSK_ERR_UNSUPPORTED.  The first (n_taps-1)/2 outputs (samples) of each channel's
 * stream are discarded once, so a centre spike with mu 0 gives the bits of the handle without the stage; the last
 * (n_taps-1)/2 samples of a call reach Mueller-Muller in the next.  Independent of qpsk_demod_set_equalizer (both may be
 * on: FLL? -> MF -> FSE -> MM -> EQ -> Costas).  May be called at any time: synchronises the handle, resets this stage
 * only (taps, window, sample counter, discard count).  With the stage on, the symbol path runs as separate kernels. */
QPSK_API int qpsk_demod_set_fractional_equalizer(qpsk_demod* d, int n_taps, float mu, float modulus);
/* the fractional stage's taps, [channels][2*n_taps]; QPSK_ERR_ARG when the stage is off */
QPSK_API int qpsk_demod_fractional_equalizer_taps(qpsk_demod* d, float* taps_iq, int64_t cap_floats);
/* DeModulate(ReadOnlySpan<float>) :345-425 -> '0'/'1' chars (not NUL-terminated).  Batch handles:
 * iq_in [channels][n_floats], bits_out [channels][cap], n_bits[channels] (same layout rule for the
 * other host entry points below). */
QPSK_API int qpsk_demod_bits(qpsk_demod* d, const float* iq_in, int64_t n_floats, char* bits_out,
                             int64_t cap, int64_t* n_bits);
/* §8f-4: DeModulate with the bits packed MSB-first, 8 per byte (BitPacker.BitsToBytes(bits, 0), HelperFunctions.cs:32-57,
 * except that a trailing incomplete byte is kept, zero-padded; n_bits[c] is the exact bit count).  packed_out is
 * [channels][cap_bytes].  One eighth of the device-to-host traffic of the char form. */
QPSK_API int qpsk_demod_bits_packed(qpsk_demod* d, const float* iq_in, int64_t n_floats, uint8_t* packed_out,
                                    int64_t cap_bytes, int64_t* n_bits);
/* DeModulateBytes :169-259 (DeModulateTextUtf8 :262-277 = this + UTF-8 decode) */
QPSK_API int qpsk_demod_bytes(qpsk_demod* d, const float* iq_in, int64_t n_floats,
                              const uint8_t* start_marker, int64_t n_start,
                              const uint8_t* end_marker, int64_t n_end,
                              uint8_t* payload_out, int64_t cap, int64_t* n_bytes);
/* DeModulateBytes on CS16 samples (interleaved int16 I, Q: the format SaveAsCs16 writes, MS/Models/HelperFunctions.cs:75-106,
 * and SDR drivers deliver, cf. TB/SDR/ModDemodOverSDR.cs:63-73): widened on the device as (float)v * scale, so the
 * host-to-device copy carries 4 bytes per complex sample instead of 8.  iq_in is [channels][n_int16]. */
QPSK_API int qpsk_demod_bytes_cs16(qpsk_demod* d, const int16_t* iq_in, int64_t n_int16, float scale,
                                   const uint8_t* start_marker, int64_t n_start, const uint8_t* end_marker, int64_t n_end,
                                   uint8_t* payload_out, int64_t cap, int64_t* n_bytes);
/* After qpsk_demod_bytes / qpsk_demod_frame_bits returned QPSK_ERR_CAPACITY (n_bytes[c] > cap for some channel): the
 * frames that call completed are still at the head of the framer ring until the next call on the handle, and this copies
 * them out ([channels][cap], n_bytes[channels] as before).  A frame that grew over several calls (the MTU-block loop of
 * TB/SDR/ModDemodOverSDR.cs:127-136) can therefore exceed a buffer sized from one call's samples without being lost. */
QPSK_API int qpsk_demod_last_payload(qpsk_demod* d, uint8_t* payload_out, int64_t cap, int64_t* n_bytes);
/* The framer half of DeModulateBytes (:182-259: carry + offset hunt :185-236, ring append and end-marker search
 * :238-258) on bits the caller already holds — what DeModulateBytes does after its DeModulate call (:177), sharing the
 * handle's framer state with qpsk_demod_bytes.  bits is HOST memory, [channels][bits_stride], one byte 0/1 per bit,
 * n_bits[channels] of them used; a channel with n_bits == 0 returns nothing and keeps its state (:179-180). */
QPSK_API int qpsk_demod_frame_bits(qpsk_demod* d, const uint8_t* bits, int64_t bits_stride, const int64_t* n_bits,
                                   const uint8_t* start_marker, int64_t n_start,
                                   const uint8_t* end_marker, int64_t n_end,
                                   uint8_t* payload_out, int64_t cap, int64_t* n_bytes);
/* deModulateConstellation :427-455 */
QPSK_API int qpsk_demod_constellation(qpsk_demod* d, const float* iq_in, int64_t n_floats,
                                      float* sym_iq_out, int64_t cap_floats, int64_t* n_sym);
/* batch, device-resident chain: d_in [channels][n_floats] (stride in floats).  Outputs per
 * channel: bits as bytes 0/1 ([channels][bits_cap], the DeModulate string after TSC strip),
 * d_n_bits[channels].  bits_cap must be even and >= qpsk_demod_bits_bound(n_floats).
 * Enqueued on `stream`, no synchronisation. */
QPSK_API int qpsk_demod_bits_dev(qpsk_demod* d, const float* d_in, int64_t n_floats, int64_t in_stride_floats,
                                 uint8_t* d_bits, int64_t bits_cap, int64_t* d_n_bits, void* stream);
/* most bits one call over n_floats can return per channel (every symbol advances >= sps-0.1 samples) */
QPSK_API int qpsk_demod_bits_bound(qpsk_demod* d, int64_t n_floats, int64_t* bits_cap);
/* DeModulateBytes, batch/device: payloads to d_payload [channels][payload_cap]; d_n_bytes[c] = payload
 * length (0 = no complete frame in this call; > payload_cap = truncated copy) */
QPSK_API int qpsk_demod_bytes_dev(qpsk_demod* d, const float* d_in, int64_t n_floats, int64_t in_stride_floats,
                                  const uint8_t* start_marker, int64_t n_start, const uint8_t* end_marker, int64_t n_end,
                                  uint8_t* d_payload, int64_t payload_cap, int64_t* d_n_bytes, void* stream);
/* deModulateConstellation, batch/device: d_sym [channels][sym_stride_floats], d_n_sym[channels] */
QPSK_API int qpsk_demod_constellation_dev(qpsk_demod* d, const float* d_in, int64_t n_floats, int64_t in_stride_floats,
                                          float* d_sym, int64_t sym_stride_floats, int* d_n_sym, void* stream);
/* per-channel loop state after the last call */
QPSK_API int qpsk_demod_loop_state(qpsk_demod* d, double* costas_theta, double* costas_freq, double* mm_mu,
                                   double* mm_integral, float* fll_phase, float* fll_freq);
/* _inFrame (:62) per channel */
QPSK_API int qpsk_demod_in_frame(qpsk_demod* d, int* in_frame);
QPSK_API int qpsk_demod_channels(const qpsk_demod* d, int* channels);
/* the CUDA device the handle was created on (every call on the handle runs there, whatever qpsk_set_device says now) */
QPSK_API int qpsk_demod_device(const qpsk_demod* d, int* ordinal);

/* ---- streaming front-end (SURVEY §8f-3): the receive loop of TB/SDR/ModDemodOverSDR.cs:116-183 ------------- */
/* That loop reads one MTU of cf32 samples into a caller-owned buffer and calls DeModulateTextUtf8 on it (:127-136).
 * A qpsk_stream keeps the call order and the per-call results (block k's payload is what the k-th
 * DeModulateBytes(block, start, end) returns on the same demodulator) but decouples the caller from the GPU:
 * push copies the block to a pinned staging slot and enqueues H2D + chain + framer + D2H on `depth` rotating slots;
 * poll returns finished payloads in push order.  The demodulator handle (single channel) stays owned by the caller,
 * must outlive the stream and must not be used directly while blocks are in flight. */
QPSK_API int qpsk_stream_create(qpsk_demod* d, int64_t max_block_floats, int64_t max_payload_bytes, int depth,
                                const uint8_t* start_marker, int64_t n_start, const uint8_t* end_marker, int64_t n_end,
                                qpsk_stream** out);
QPSK_API int qpsk_stream_destroy(qpsk_stream* s);
/* one block of interleaved cf32 (n_floats even, <= max_block_floats); returns without waiting for the GPU unless all
 * `depth` slots are still in flight */
QPSK_API int qpsk_stream_push(qpsk_stream* s, const float* iq, int64_t n_floats);
/* the same block as CS16 (interleaved int16 I,Q — MS/Models/HelperFunctions.cs:75-106 writes this format); widened on the
 * device as (float)v * scale, so PCIe carries 4 bytes per complex sample instead of 8 */
QPSK_API int qpsk_stream_push_cs16(qpsk_stream* s, const int16_t* iq, int64_t n_int16, float scale);
/* next block's result in push order.  *have_block = 0: nothing finished yet (wait = 0) or nothing outstanding.
 * *n_bytes is the payload length of that block (0 = no complete frame in it, like Array.Empty :258);
 * > cap -> QPSK_ERR_CAPACITY with the block consumed. */
QPSK_API int qpsk_stream_poll(qpsk_stream* s, int wait, uint8_t* payload_out, int64_t cap, int64_t* n_bytes, int* have_block);
QPSK_API int qpsk_stream_pending(qpsk_stream* s, int64_t* pushed, int64_t* polled);
QPSK_API int qpsk_stream_flush(qpsk_stream* s);              /* wait until every pushed block has finished */

/* CS16 <-> cf32.  to_cs16 follows SaveAsCs16 (HelperFunctions.cs:75-106): scale by short.MaxValue / max(|re|,|im|) in
 * fp64 (max < 1e-12 -> 1), clamp to [short.MinValue, short.MaxValue], truncate toward zero; empty input -> QPSK_ERR_ARG
 * (:79-80).  *max_abs receives the normalisation factor (needed to undo it).  to_cf32: out = (float)v * scale. */
QPSK_API int qpsk_cf32_to_cs16(const float* iq, int64_t n_floats, int16_t* out, float* max_abs);
QPSK_API int qpsk_cs16_to_cf32(const int16_t* in, int64_t n_int16, float scale, float* out);
QPSK_API int qpsk_cf32_to_cs16_dev(const float* d_in, int64_t n_floats, int16_t* d_out, float* d_max_abs, void* stream);
QPSK_API int qpsk_cs16_to_cf32_dev(const int16_t* d_in, int64_t n_int16, float scale, float* d_out, void* stream);

/* ---- full receive chain (SURVEY §8f-2): TB/Simulated/testFullDemodChain.cs:14-116, repaired ------- */
/* FLL -> RRC matched filter -> Mueller-Muller -> Costas wired as that test does by hand (:22-45, :73-110),
 * every block parameter explicit (upstream the test no longer constructs: SURVEY §4).  The three outputs are
 * the payloads of the ZMQ topics the test publishes — raw little-endian cf32, byte-identical to these float
 * buffers (:88-108): "baseband" = FLL output (one per input sample), "baseband_PostSymbolSync" = MM symbols,
 * "baseband_PostSymbolSyncPostCostas" = Costas output.  State persists across calls (any chunking gives the
 * same three streams). */
typedef struct qpsk_chain_params {
  int sample_rate, symbol_rate;      /* matched filter = RRC(rrc_span, rrc_alpha, sample_rate, symbol_rate) :22 */
  double rrc_span, rrc_alpha;
  float fll_sps, fll_rolloff;        /* FLLBandEdgeFilter(sps, rolloff, size, bandwidth) :23                    */
  int fll_size;
  float fll_bw;
  double mm_sps, mm_kp, mm_ki;       /* MuellerMuller(sps, Kp, Ki) :35-39                                       */
  double costas_sample_rate, costas_bw_hz, costas_damping; /* CostasLoopQpsk(SymbolRate, SymbolRate/10) :45    */
} qpsk_chain_params;
/* the literal values of testFullDemodChain.cs:18-45 (fs 10 MHz, Rs fs/30, span 11, alpha .9, FLL(30,.9,10,.1)) */
QPSK_API int qpsk_chain_default_params(qpsk_chain_params* p);
QPSK_API int qpsk_chain_create(const qpsk_chain_params* p, int channels, qpsk_chain** out);
QPSK_API int qpsk_chain_destroy(qpsk_chain* c);
/* matched-filter arithmetic: QPSK_FIR_FAST (default) or QPSK_FIR_EXACT (the reference's summation order) */
QPSK_API int qpsk_chain_set_fir_mode(qpsk_chain* c, int mode);
/* floats one call of n_floats input can emit per channel on the two symbol outputs */
QPSK_API int qpsk_chain_symbols_bound(const qpsk_chain* c, int64_t n_floats, int64_t* cap_floats);
/* host pointers: iq_in / baseband_out [channels][n_floats]; sync_out / costas_out [channels][sym_cap_floats];
 * n_sym[channels] complex symbols produced */
QPSK_API int qpsk_chain_process(qpsk_chain* c, const float* iq_in, int64_t n_floats, float* baseband_out, float* sync_out,
                                float* costas_out, int64_t sym_cap_floats, int* n_sym);
/* device pointers, strides in floats (even), d_n_sym int[channels] in device memory */
QPSK_API int qpsk_chain_process_dev(qpsk_chain* c, const float* d_in, int64_t n_floats, int64_t in_stride, float* d_baseband,
                                    int64_t bb_stride, float* d_sync, int64_t sync_stride, float* d_costas,
                                    int64_t costas_stride, int* d_n_sym, void* stream);
/* per-channel loop state (any pointer may be NULL) */
QPSK_API int qpsk_chain_loop_state(qpsk_chain* c, float* fll_phase, float* fll_freq, double* mm_mu, double* costas_theta,
                                   double* costas_freq);

/* ---- synthetic channel (SURVEY §8f-1): NCO pair + AWGN + static multipath ------------------- */
/* NCO: TB/Simulated/LocalOscilator.cs:5-194; noise: TB/HelperModels.cs:17-45; System.Random is
 * replaced by the counter RNG of DESIGN.md.  Channel c uses RNG streams 4c (tx NCO), 4c+1 (rx NCO),
 * 4c+2 (noise), 4c+3 (payload bits). */
typedef struct qpsk_chan_params {
  double tx_freq_hz, rx_freq_hz, sample_rate_hz;
  double tx_ppm, rx_ppm, tx_phase0, rx_phase0;
  float noise_dbfs;       /* <= -300: no noise                                                    */
  int mode;               /* 0: x*(tx*conj(rx)) (testAtDataLevel.cs:39-42); 1: ((x+n)*tx)*conj(rx)
                             (testFullDemodChain.cs:73)                                           */
  int n_paths;            /* 0 = no multipath; else <= 4 paths                                    */
  float path_gain_iq[8];
  int path_delay[4];
  uint64_t seed;
} qpsk_chan_params;
QPSK_API int qpsk_chan_create(const qpsk_chan_params* p, int channels, int first_channel, qpsk_chan** out);
QPSK_API int qpsk_chan_destroy(qpsk_chan* c);
/* y[c][n] = channel_c(x[c][n]); state (NCO phase, drift, counters) persists across calls.
 * x_stride 0 = the same burst for every channel. */
QPSK_API int qpsk_chan_apply_dev(qpsk_chan* c, const float* d_x, int64_t n_floats, int64_t x_stride_floats,
                                 float* d_y, int64_t y_stride_floats, void* stream);
QPSK_API int qpsk_chan_apply(qpsk_chan* c, const float* x, int64_t n_floats, float* y);
/* uniform(-1,1) fp32 fill from the counter RNG: out[k] = (float)(2*u(seed,stream,first+k)-1) */
QPSK_API int qpsk_fill_uniform_dev(uint64_t seed, uint64_t stream_id, int64_t first, int64_t n, float* d_out, void* stream);
/* random payload bytes: out[c][k] = top byte of rng(seed, 4*(first_channel+c)+3, k) */
QPSK_API int qpsk_fill_bytes_dev(uint64_t seed, int first_channel, int channels, int64_t n_bytes, uint8_t* d_out, void* stream);

/* bits[c][8k+j] = bit (7-j) of bytes[c][k] as bytes 0/1 (BitPacker.BytesToBitString, HelperFunctions.cs:14-29) */
QPSK_API int qpsk_unpack_bits_dev(const uint8_t* d_bytes, int64_t n_bytes, int64_t bytes_stride, int channels,
                                  uint8_t* d_bits, int64_t bits_stride, void* stream);

/* ---- K6  per-channel BER counters ---------------------------------------------------------- */
/* bytes 0/1 -> MSB-first packed bytes per channel (n_bits[c] bits each, at most max_bits; trailing partial byte zero-padded) */
QPSK_API int qpsk_pack_bits_dev(const uint8_t* d_bits, int64_t bits_stride, const int64_t* d_n_bits, int64_t max_bits,
                                int channels, uint8_t* d_packed, int64_t packed_stride, void* stream);
/* bits as bytes 0/1.  errors[c] = Hamming distance over min(n_rx[c], n_ref) bits + max(0, n_ref-n_rx[c])
 * (bits that never arrived count as errors, extra trailing bits are ignored);
 * counters[c] = {errors, n_ref}.  ref_stride 0 = one reference for all channels. */
QPSK_API int qpsk_ber_count_dev(const uint8_t* d_rx_bits, int64_t rx_stride, const int64_t* d_n_rx,
                                const uint8_t* d_ref_bits, int64_t ref_stride, int64_t n_ref,
                                int channels, uint32_t* d_counters, void* stream);

/* ---- the one collective (SURVEY §8e): all-gather of the per-channel BER counters over NCCL ------------------------ */
/* Channels are independent and sharded in contiguous blocks, one block per GPU (channel c on rank floor(c*G/C)); nothing is
 * exchanged on the data path.  After a run each rank holds {errors, bits}[channels_local] from qpsk_ber_count_dev; these
 * calls collect the whole table on every rank.  One communicator per process (or thread) and GPU: rank 0 makes the id,
 * ships its QPSK_COMM_ID_BYTES to the other ranks by any means (a file, a socket, MPI, torch.distributed's store), and
 * all ranks call qpsk_comm_create — a collective — on the device chosen with qpsk_set_device.  NCCL is loaded with
 * dlopen("libnccl.so.2"); without it these calls return QPSK_ERR_UNSUPPORTED and nothing else in the library is affected. */
typedef struct qpsk_comm qpsk_comm;
#define QPSK_COMM_ID_BYTES 128
QPSK_API int qpsk_comm_unique_id(uint8_t* id, int cap);                       /* ncclGetUniqueId */
QPSK_API int qpsk_comm_create(const uint8_t* id, int n_ranks, int rank, qpsk_comm** out);   /* ncclCommInitRank */
QPSK_API int qpsk_comm_destroy(qpsk_comm* c);
/* what the communicator itself reports (ncclCommCount / ncclCommUserRank) and the NCCL version in use */
QPSK_API int qpsk_comm_info(qpsk_comm* c, int* n_ranks, int* rank, int* nccl_version);
/* d_counters: this rank's uint32 {errors, bits}[channels_local] in device memory; channels_max = the largest block of any
 * rank (blocks differ by at most one channel when G does not divide C).  d_all (device, every rank):
 * [n_ranks][channels_max][2], rank r's block at row r*channels_max, rows past a rank's own count {0, 0}.  Enqueued on
 * `stream` (NULL = the communicator's own), no synchronisation. */
QPSK_API int qpsk_ber_gather_dev(qpsk_comm* c, const uint32_t* d_counters, int channels_local, int channels_max,
                                 uint32_t* d_all, void* stream);
/* the same into host memory (all_host[n_ranks*channels_max*2]); d_counters must be complete when it is called */
QPSK_API int qpsk_ber_gather(qpsk_comm* c, const uint32_t* d_counters, int channels_local, int channels_max, uint32_t* all_host);

/* ---- measurement helpers ------------------------------------------------------------------- */
/* FP32 FMA-pipe peak (TFLOP/s) by a register-resident FFMA micro-benchmark, for the roofline */
QPSK_API int qpsk_measure_fma_peak(double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* QPSKCUDA_H_ */
