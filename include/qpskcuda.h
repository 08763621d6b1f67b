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
/* filter_size 1..1430: every size must run in the generic kernel, whose ring of filter_size past outputs per stream lives
   in shared memory (16 streams per CTA, within 200 KiB).  Larger sizes return QPSK_ERR_UNSUPPORTED, here, in
   qpsk_fll_create_batch and in qpsk_chain_create (fll_size). */
QPSK_API int qpsk_fll_create(float sps, float rolloff, int filter_size, float bandwidth, qpsk_fll** out);
QPSK_API int qpsk_fll_create_batch(float sps, float rolloff, int filter_size, float bandwidth,
                                   int channels, qpsk_fll** out);
QPSK_API int qpsk_fll_destroy(qpsk_fll* f);
/* Process(ReadOnlySpan<float>, Span<float>) :64-87 */
QPSK_API int qpsk_fll_process(qpsk_fll* f, const float* iq_in, float* iq_out, int64_t n_floats,
                              int64_t out_cap_floats);
/* device memory (8-byte aligned, else QPSK_ERR_ARG), strides in floats */
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
/* device memory (8-byte aligned, else QPSK_ERR_ARG), strides in floats; d_n_sym[channels] symbols written */
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
/* batch/device (8-byte aligned, else QPSK_ERR_ARG): n_sym[channels] valid complex samples per channel (NULL = n_floats/2
 * for all) */
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
/* device memory (8-byte aligned, else QPSK_ERR_ARG), strides in floats; d_n_sym[channels] valid complex symbols per
 * channel (NULL = n_floats/2 for all) */
QPSK_API int qpsk_eq_process_dev(qpsk_eq* eq, const float* d_in, float* d_out, int64_t n_floats, int64_t in_stride_floats,
                                 int64_t out_stride_floats, const int* d_n_sym, void* stream);
/* taps [channels][2*n_taps] interleaved IQ; get: cap_floats < channels*2*n_taps -> QPSK_ERR_CAPACITY; set: n_floats must be
 * exactly channels*2*n_taps (else QPSK_ERR_ARG), every value finite (else QPSK_ERR_RANGE) */
QPSK_API int qpsk_eq_get_taps(qpsk_eq* eq, float* taps_iq, int64_t cap_floats);
QPSK_API int qpsk_eq_set_taps(qpsk_eq* eq, const float* taps_iq, int64_t n_floats);

/* ---- polyphase analysis channelizer ------------------------------------------------------------------------ */
/* Not in the reference (it receives one carrier per stream); the block that splits ONE wideband capture holding M carriers
 * on a frequency grid into the [channels][samples] batch the demodulator takes: a critically sampled polyphase filter-bank
 * (PFB) analysis channelizer, GNU Radio's pfb_channelizer_ccf without oversampling.
 * Parameters: real prototype taps h[0..n_taps-1]; M channels, a power of two 2..1024; the taps are zero-padded at the end
 * to L = P*M with P = ceil(n_taps/M) taps per branch, 1 <= P <= 32 (outside these limits: QPSK_ERR_UNSUPPORTED; n_taps <= 0:
 * QPSK_ERR_ARG; a non-finite tap: QPSK_ERR_RANGE).
 * Blocks: x[n] counts samples since creation or the last reset, x[n] = 0 for n < 0.  Output m exists once block m, samples
 * mM .. mM+M-1, is complete.  With N = mM + M - 1:
 *   y_k[m] = sum_{i=0}^{L-1} h[i] * e^{+j 2 pi k i / M} * x[N - i],   k = 0..M-1.
 * Channel k is the band centred at +k/M cycles per input sample, rows in natural order (no fftshift: k >= M/2 are the
 * negative frequencies k - M).  No 1/M factor: a prototype with sum h = 1 passes a carrier centred on channel k with unit
 * gain, so the CMA `modulus 1.0` convention holds after the channelizer.  Against "mix down by k/M, filter with h, keep
 * every M-th sample (n = N)", channel k carries the constant phase e^{-j 2 pi k / M}.
 * Computation (the equivalent polyphase form): v_r[m] = sum_{q=0}^{P-1} h[qM + r] * x[(m - q)M + M - 1 - r], accumulated
 * in increasing q, then y_k[m] = sum_r v_r[m] * w^{kr}, w = e^{j 2 pi / M}, by an in-place radix-2/radix-2^2 FFT.  fp32 with
 * FMA; twiddles from an fp64 table rounded to fp32.  Against an fp64 evaluation of the definition max|err| <= 1e-5 max|y|,
 * and per output (re and im, every channel k of block m), with u = 2^-24, gamma_n = nu / (1 - nu), S = log2 M and
 * eta = 4u + O(u^2): |err| <= (1+eta)^S sum_r gamma_P |(sum_q |h||x.re|, sum_q |h||x.im|)| + ((1+eta)^S - 1) sum_r |v_r[m]|
 * (derivation: tests/bank_bounds.py).
 * State: the last (P-1) complete blocks and the pending = (samples so far) mod M samples of the open block.  Any chunking of
 * a stream (chunks shorter than M, empty calls, any pointer alignment that results) gives the same outputs bit for bit.
 * A call of n samples gives floor((pending + n) / M) outputs per channel, known to the host without reading the device. */
typedef struct qpsk_pfb qpsk_pfb;
/* Kaiser-windowed sinc prototype, host fp64, unit DC gain; L = taps_per_branch*channels taps, cutoff in cycles per input
 * sample (0 < cutoff < 0.5, else QPSK_ERR_RANGE), beta from atten_db (finite, >= 0) by Kaiser's formula.  Same as
 * scipy.signal.firwin(L, 2*cutoff, window=("kaiser", kaiser_beta(atten_db)), scale=True).  channels / taps_per_branch
 * outside the limits above: QPSK_ERR_UNSUPPORTED.  out==NULL or cap too small: *n still set (like qpsk_rrc_taps). */
QPSK_API int qpsk_pfb_taps(int channels, int taps_per_branch, double cutoff, double atten_db, double* out, int cap, int* n);
QPSK_API int qpsk_pfb_create(const float* taps, int n_taps, int channels, qpsk_pfb** out);
QPSK_API int qpsk_pfb_destroy(qpsk_pfb* p);
/* back to the state at creation: no history, no pending samples.  Waits for the handle's own stream only: qpsk_pfb_process_dev
 * calls enqueued on another stream must have completed before the reset (synchronise that stream first). */
QPSK_API int qpsk_pfb_reset(qpsk_pfb* p);
/* host memory: iq_in n_floats (even, else QPSK_ERR_ARG) of ONE wideband stream -> iq_out [channels][out_stride_floats];
 * *n_out_floats = floats written per channel (set on QPSK_ERR_CAPACITY too); out_stride_floats < *n_out_floats ->
 * QPSK_ERR_CAPACITY, nothing consumed.  Floats of a row past *n_out_floats are not written. */
QPSK_API int qpsk_pfb_process(qpsk_pfb* p, const float* iq_in, int64_t n_floats, float* iq_out,
                              int64_t out_stride_floats, int64_t* n_out_floats);
/* device memory (8-byte aligned, else QPSK_ERR_ARG), out_stride_floats even: the [channels][out_stride] rows
 * qpsk_demod_bits_dev / qpsk_demod_bytes_dev read with in_stride = out_stride; pass both calls the same stream (NULL means
 * each handle's own stream, and nothing then orders the demodulator's reads after these writes).  Enqueued on `stream`;
 * the handle's state advances at enqueue, so calls on one handle must run in issue order. */
QPSK_API int qpsk_pfb_process_dev(qpsk_pfb* p, const float* d_in, int64_t n_floats, float* d_out,
                                  int64_t out_stride_floats, int64_t* n_out_floats, void* stream);

/* ---- digital down-converter bank ---------------------------------------------------------------------------- */
/* Not in the reference; the front end for carriers at arbitrary frequencies in ONE wideband capture: K digital
 * down-converters (mix by -f_k, lowpass with a shared real prototype, keep every D-th sample) sharing one pass over the
 * input, GNU Radio's freq_xlating_fir_filter_ccf once per carrier.  Unlike the PFB channelizer the carriers need no grid,
 * any subset of frequencies is computed, and the output rate is 1/D whatever K is.
 * Parameters: real taps h[0..n_taps-1], 1 <= n_taps <= 4096; K channels, 1 <= K <= 2048; decimation D, 1 <= D <= 1024;
 * frequencies f_k in cycles per input sample, each finite and in [-0.5, 0.5) (outside the limits on K, D and n_taps:
 * QPSK_ERR_UNSUPPORTED; n_taps <= 0: QPSK_ERR_ARG; a non-finite tap or a bad frequency: QPSK_ERR_RANGE).
 * Phase words: inc_k = nearbyint(ldexp(f_k, 64)) mod 2^64 (uint64); the phase of stream sample n is phi_k(n) = inc_k * n
 * mod 2^64, exact unsigned 64-bit arithmetic, n counting samples since creation or the last reset.  No phase is
 * accumulated in floating point, so it is chunk-invariant and identical on the host, the device and in a reference.
 * Output: x[n] = 0 for n < 0.  Output m exists once samples up to n_m = mD + D - 1 have arrived; with N = n_taps
 *   y_k[m] = sum_{i=0}^{N-1} h[i] * x[n_m - i] * e^{-j 2 pi phi_k(n_m - i) / 2^64}
 * ("mix down by f_k, filter with h, keep every D-th sample").  No 1/D factor: a prototype with sum h = 1 passes a tuned
 * carrier with unit gain and no rotation, so the CMA `modulus 1.0` convention holds after the bank.
 * Computation (exact in the phase words, phi(n - i) = phi(n) - phi(i) mod 2^64): u_k[m] = sum_i g_k[i] x[n_m - i] with
 * rotated taps g_k[i] = h[i] e^{+j 2 pi phi_k(i) / 2^64} formed on the host in fp64 and rounded to fp32, then
 * y_k[m] = u_k[m] e^{-j 2 pi phi_k(n_m) / 2^64}.  fp32 with FMA; against an fp64 evaluation of the definition
 * max|err| <= 1e-5 max|y| over a call's output, and per output (re and im), with u = 2^-24 and A = sum_i |h[i]|
 * (|x[n_m - i].re| + |x[n_m - i].im|): |err| <= about sqrt2 (N + 1) u A + (5u + pi (2^-31 + 2^-25)) |u_k[m]| (the exact
 * constants and their derivation: tests/bank_bounds.py).
 * Relation to the PFB channelizer: with D = M and f_k = k/M (k >= M/2 taken as k - M), row k of the bank equals row k of
 * qpsk_pfb with the same prototype times e^{+j 2 pi k / M}.  For a full grid the PFB is the cheaper block.
 * State: the last N-1 input samples, the pending = (samples so far) mod D samples of the open block and the 64-bit sample
 * counter.  Any chunking of a stream (chunks shorter than D, empty calls, any pointer alignment that results) gives the
 * same outputs bit for bit.  A call of n samples gives floor((pending + n) / D) outputs per channel, known to the host. */
typedef struct qpsk_ddc qpsk_ddc;
QPSK_API int qpsk_ddc_create(const float* taps, int n_taps, const double* freqs, int channels, int decim, qpsk_ddc** out);
QPSK_API int qpsk_ddc_destroy(qpsk_ddc* p);
/* back to the state at creation: no history, no pending samples, counter 0.  Waits for the handle's own stream only:
 * qpsk_ddc_process_dev calls enqueued on another stream must have completed before the reset. */
QPSK_API int qpsk_ddc_reset(qpsk_ddc* p);
/* host memory: iq_in n_floats (even, else QPSK_ERR_ARG) of ONE wideband stream -> iq_out [channels][out_stride_floats];
 * *n_out_floats = floats written per channel (set on QPSK_ERR_CAPACITY too); out_stride_floats < *n_out_floats ->
 * QPSK_ERR_CAPACITY, nothing consumed.  Floats of a row past *n_out_floats are not written. */
QPSK_API int qpsk_ddc_process(qpsk_ddc* p, const float* iq_in, int64_t n_floats, float* iq_out,
                              int64_t out_stride_floats, int64_t* n_out_floats);
/* device memory (8-byte aligned, else QPSK_ERR_ARG), out_stride_floats even: the [channels][out_stride] rows
 * qpsk_demod_bits_dev / qpsk_demod_bytes_dev read with in_stride = out_stride; pass both calls the same stream (NULL means
 * each handle's own stream, and nothing then orders the demodulator's reads after these writes).  Enqueued on `stream`;
 * the handle's state advances at enqueue, so calls on one handle must run in issue order. */
QPSK_API int qpsk_ddc_process_dev(qpsk_ddc* p, const float* d_in, int64_t n_floats, float* d_out,
                                  int64_t out_stride_floats, int64_t* n_out_floats, void* stream);

/* ---- feed-forward AGC ----------------------------------------------------------------------------------------- */
/* Not in the reference (its chain assumes unit amplitude); the level normaliser for a batch of channels that arrive at
 * different levels, e.g. the carriers of one capture after qpsk_pfb / qpsk_ddc.  GNU Radio's feedforward_agc_cc made
 * causal: one gain per sample from the peak envelope of a W-sample window that looks ahead of the sample it scales.
 * Parameters: window W, 1..4096 (else QPSK_ERR_UNSUPPORTED); ref and max_gain finite and > 0 (else QPSK_ERR_RANGE);
 * channels >= 1 (else QPSK_ERR_RANGE).
 * Definition, per channel, x[n] counting samples since creation or the last reset, x[n] = 0 for n < 0:
 *   env(v) = fmaxf(fabsf(v.re), fabsf(v.im))                                  (exact)
 *   m[n]   = fmaxf over {0, env(x[n - i]) : i = 0..W-1}                         (exact; a NaN envelope is ignored)
 *   g[n]   = fminf(ref / m[n], max_gain)                                       (one rounding; m = 0 gives max_gain)
 *   y[n]   = (x[n-W+1].re * g[n], x[n-W+1].im * g[n])                          (one rounding each)
 * so the window of output n runs from the sample it scales, x[n-W+1], W-1 samples ahead to x[n]: the output stream is the
 * input delayed by W-1 samples (its first W-1 outputs scale the zero history).  fp32, no FMA anywhere, so the GPU equals
 * any CPU restatement bit for bit (a NaN output is NaN; its sign and payload are not specified).  Scaling the input by 2^k changes no output bit unless max_gain binds or a value
 * leaves the normal range.  State: the last W-1 samples and the last gain of each channel.  Any chunking of a stream
 * (empty calls, chunks shorter than W) gives the same outputs bit for bit.  One output per input sample. */
typedef struct qpsk_agc qpsk_agc;
QPSK_API int qpsk_agc_create_batch(int window, float ref, float max_gain, int channels, qpsk_agc** out);
QPSK_API int qpsk_agc_destroy(qpsk_agc* p);
/* back to the state at creation: zero history, every last gain max_gain.  Waits for the handle's own stream only:
 * qpsk_agc_process_dev calls enqueued on another stream must have completed before the reset. */
QPSK_API int qpsk_agc_reset(qpsk_agc* p);
/* host memory, iq_in / iq_out [channels][n_floats]; odd n_floats -> QPSK_ERR_ARG, out_cap_floats < n_floats ->
 * QPSK_ERR_CAPACITY.  A refused call consumes nothing. */
QPSK_API int qpsk_agc_process(qpsk_agc* p, const float* iq_in, float* iq_out, int64_t n_floats, int64_t out_cap_floats);
/* device memory (8-byte aligned, else QPSK_ERR_ARG), strides in floats (even; in_stride_floats >= n_floats, else
 * QPSK_ERR_ARG; out_stride_floats < n_floats -> QPSK_ERR_CAPACITY); d_out must not overlap d_in.  Enqueued on `stream`
 * (NULL = the handle's own); the state advances at enqueue, so calls on one handle must run in issue order.  Floats of a
 * row past n_floats are not written. */
QPSK_API int qpsk_agc_process_dev(qpsk_agc* p, const float* d_in, float* d_out, int64_t n_floats, int64_t in_stride_floats,
                                  int64_t out_stride_floats, void* stream);
/* gain of each channel's last output, gain[channels] (cap < channels -> QPSK_ERR_CAPACITY); synchronises the handle's own
 * stream.  The _dev form copies them to d_gain[channels] on `stream` (NULL = the handle's own) in stream order. */
QPSK_API int qpsk_agc_gain(qpsk_agc* p, float* gain, int64_t cap);
QPSK_API int qpsk_agc_gain_dev(qpsk_agc* p, float* d_gain, void* stream);

/* ---- rational resampler ------------------------------------------------------------------------------------- */
/* Not in the reference; moves a batch of channel streams between sample rates that are not integer multiples of each
 * other (a fixed ADC / DAC rate against the symbol rate), GNU Radio's rational_resampler_ccf once per channel: interpolate
 * by L, filter with a real prototype, decimate by M.
 * Parameters: real taps h[0..N-1], 1 <= N <= 16384; interpolation L and decimation M, each 1..1024 (not necessarily
 * coprime); P = ceil(N / L) taps per branch, P <= 64; channels 1..16384 (outside these limits: QPSK_ERR_UNSUPPORTED;
 * N <= 0: QPSK_ERR_ARG; a non-finite tap: QPSK_ERR_RANGE).
 * Definition, per channel, x[n] counting input samples since creation or the last reset, x[n] = 0 for n < 0, x_up = x
 * zero-stuffed by L (x_up[nL] = x[n], zero elsewhere):
 *   y[m] = sum_{i=0}^{N-1} h[i] * x_up[mM - i]                       (scipy.signal.upfirdn(h, x, L, M) taken literally)
 * Computation (the polyphase form): n_m = floor(mM / L), phi_m = mM mod L, exact integer arithmetic on 64-bit counters (no
 * position is accumulated in floating point), and y[m] = sum_{q=0}^{P-1} h[phi_m + qL] * x[n_m - q] with h zero past N,
 * accumulated in increasing q with fp32 FMA, re and im separately.  Against an fp64 evaluation of the definition
 * max|err| <= 1e-5 max|y| over a call's output, and per output |err.re| <= gamma_P sum_q |h[phi_m + qL]| |x[n_m - q].re|
 * (the same for im), gamma_P = Pu / (1 - Pu), u = 2^-24.
 * No L factor: a prototype with sum h = L (e.g. L * firwin(..., scale=True)) passes a carrier with unit gain, so the CMA
 * `modulus 1.0` convention holds after the resampler.
 * Output m exists once x[n_m] has arrived: after n_in inputs there are n_in == 0 ? 0 : floor((n_in L - 1) / M) + 1
 * outputs, and a call's count is that difference, known to the host without reading the device.
 * State: the last P-1 input samples of each channel and the input and output counters.  Any chunking of a stream (empty
 * calls, chunks shorter than M / L, any sample offset) gives the same outputs bit for bit, and row c of a batch equals a
 * one-channel handle fed that row, bit for bit. */
typedef struct qpsk_resamp qpsk_resamp;
QPSK_API int qpsk_resamp_create(const float* taps, int n_taps, int interp, int decim, int channels, qpsk_resamp** out);
QPSK_API int qpsk_resamp_destroy(qpsk_resamp* p);
/* back to the state at creation: zero history, counters 0.  Waits for the handle's own stream only:
 * qpsk_resamp_process_dev calls enqueued on another stream must have completed before the reset. */
QPSK_API int qpsk_resamp_reset(qpsk_resamp* p);
/* host memory: iq_in [channels][n_floats] (n_floats even, else QPSK_ERR_ARG) -> iq_out [channels][out_stride_floats];
 * *n_out_floats = floats written per channel (set on QPSK_ERR_CAPACITY too); out_stride_floats < *n_out_floats ->
 * QPSK_ERR_CAPACITY, nothing consumed.  Floats of a row past *n_out_floats are not written. */
QPSK_API int qpsk_resamp_process(qpsk_resamp* p, const float* iq_in, int64_t n_floats, float* iq_out,
                                 int64_t out_stride_floats, int64_t* n_out_floats);
/* device memory (8-byte aligned, else QPSK_ERR_ARG), strides in floats (even; in_stride_floats >= n_floats, else
 * QPSK_ERR_ARG; out_stride_floats < *n_out_floats -> QPSK_ERR_CAPACITY with *n_out_floats set and nothing consumed); the
 * rows written must not overlap the rows read (QPSK_ERR_ARG).  d_out's rows are the [channels][out_stride] rows
 * qpsk_demod_bytes_dev reads with in_stride = out_stride, and d_in's can be the rows qpsk_ddc_process_dev writes.
 * Enqueued on `stream` (NULL = the handle's own); the state advances at enqueue, so calls on one handle must run in issue
 * order.  Floats of a row past *n_out_floats are not written. */
QPSK_API int qpsk_resamp_process_dev(qpsk_resamp* p, const float* d_in, int64_t n_floats, int64_t in_stride_floats,
                                     float* d_out, int64_t out_stride_floats, int64_t* n_out_floats, void* stream);

/* ---- convolutional code: K = 7, rate 1/2, encoder and soft-decision Viterbi decoder ---------------------------------- */
/* Not in the reference; forward error correction for the coded receive path
 *   qpsk_demod_constellation_dev -> qpsk_viterbi_decode_dev -> qpsk_demod_frame_bits_dev.
 * The code (fixed): register s, the current input bit at bit 6 and the oldest at bit 0; each input bit emits the pair
 * (c0, c1) = (parity(s & 0171), parity(s & 0133)) (octal), c0 first.  An impulse encodes to 11 10 11 11 00 01 11.  One
 * pair is one QPSK symbol: c0 is the dibit's first bit (the I bit without differential encoding, the first bit of
 * DibitToDelta with it), so one trellis step is one symbol.  Bits are bytes 0/1 ([channels][stride]), the format of
 * qpsk_unpack_bits_dev and qpsk_ber_count_dev.  1..16384 channels (else QPSK_ERR_UNSUPPORTED).
 * Encoder: the six-bit register of each channel persists across calls (zero at creation and reset), so any chunking of a
 * stream gives the same bits.  A nonzero input byte is a 1. */
typedef struct qpsk_conv qpsk_conv;
QPSK_API int qpsk_conv_create(int channels, qpsk_conv** out);
QPSK_API int qpsk_conv_destroy(qpsk_conv* p);
QPSK_API int qpsk_conv_reset(qpsk_conv* p);
/* host: bits [channels][n_bits] -> out [channels][2*n_bits] */
QPSK_API int qpsk_conv_encode(qpsk_conv* p, const uint8_t* bits, int64_t n_bits, uint8_t* out);
/* device: d_bits [channels][bits_stride] (bits_stride >= n_bits, else QPSK_ERR_ARG) -> d_out [channels][out_stride]
 * (out_stride < 2*n_bits: QPSK_ERR_CAPACITY, nothing consumed); enqueued on `stream` (NULL = the handle's own) */
QPSK_API int qpsk_conv_encode_dev(qpsk_conv* p, const uint8_t* d_bits, int64_t n_bits, int64_t bits_stride, uint8_t* d_out,
                                  int64_t out_stride, void* stream);
/* Decoder, per channel; every rule below is exact, and the GPU is bit-identical to tests/fec_oracle.py.
 * 1. Soft values, int8, positive = bit 1: q(v) = clamp(rint_half_even(v), -127, 127) (NaN -> 0); every product and sum
 *    is a separately rounded fp32 operation (no FMA contraction).
 *      coherent:      s0 = q(scale*I), s1 = q(scale*Q)
 *      differential:  z = y_k conj(y_{k-1}), re = yr*pr + yi*pi, im = yi*pr - yr*pi;
 *                     s0 = q(-(scale*(re+im))), s1 = q(scale*(im-re))   (soft form of 00->+1, 01->+j, 11->-1, 10->-j)
 *    y_{k-1} is carried across calls; the first symbol a handle sees after create, reset or flush yields no step (the
 *    reference receiver drops its first symbol too).
 * 2. Add-compare-select over the 64 states S (the last six inputs, the newest at bit 5): branch metric
 *    sum_i (c_i ? -s_i : s_i), smaller is better; predecessors of a state in increasing state order, a tie keeps the lower;
 *    every metric starts at 0 (unknown start state); integer metrics, renormalised by subtracting the minimum every 32 steps.
 * 3. Decisions, B = 32, D = 64: once absolute step (k+1)*B + D - 1 of a channel has been processed, the bits of steps
 *    [k*B, (k+1)*B) are read off the survivor path of the best state at that step (minimum metric, lowest state on ties).
 *    A flush reads every step not yet emitted off the best state at the last step, then resets the handle.
 * Default scales for symbols at unit amplitude (Costas output; the opt-in AGC stage delivers that level), from an oracle
 * BER sweep (DESIGN.md §3 K13).  In differential mode z scales with the square of the amplitude. */
#define QPSK_VITERBI_SCALE_COHERENT 32.0f
#define QPSK_VITERBI_SCALE_DIFFERENTIAL 24.0f
typedef struct qpsk_viterbi qpsk_viterbi;
/* differential: 0 / 1; scale finite and > 0 (else QPSK_ERR_RANGE) */
QPSK_API int qpsk_viterbi_create(int channels, int differential, float scale, qpsk_viterbi** out);
QPSK_API int qpsk_viterbi_destroy(qpsk_viterbi* p);
/* back to the state at creation.  Waits for the handle's own stream only. */
QPSK_API int qpsk_viterbi_reset(qpsk_viterbi* p);
/* the most bits one decode or flush call over at most max_sym symbols per channel can emit: max_sym + 96 rounded down
 * to even (whole blocks of 32, plus the up to 95 steps a flush adds) */
QPSK_API int qpsk_viterbi_bits_bound(const qpsk_viterbi* p, int64_t max_sym, int64_t* cap);
/* Device: d_sym [channels][sym_stride_floats] cf32 and int d_n_sym[channels] (what qpsk_demod_constellation_dev writes;
 * ragged, 0 allowed; a count past sym_stride_floats/2 is read as sym_stride_floats/2) -> decided bits d_bits
 * [channels][bits_cap] and int64 d_n_bits[channels], the layout qpsk_ber_count_dev and qpsk_demod_frame_bits_dev read.
 * Pointers 8-byte aligned and strides even (else QPSK_ERR_ARG); bits_cap < qpsk_viterbi_bits_bound(sym_stride_floats/2):
 * QPSK_ERR_CAPACITY before any state advances.  Enqueued on `stream` (NULL = the handle's own); state lives on the device,
 * so calls on one handle must run in issue order.  Bytes of a row past d_n_bits[c] are not written. */
QPSK_API int qpsk_viterbi_decode_dev(qpsk_viterbi* p, const float* d_sym, int64_t sym_stride_floats, const int* d_n_sym,
                                     uint8_t* d_bits, int64_t bits_cap, int64_t* d_n_bits, void* stream);
/* decode the call's symbols, emit every step not yet emitted, reset the handle */
QPSK_API int qpsk_viterbi_flush_dev(qpsk_viterbi* p, const float* d_sym, int64_t sym_stride_floats, const int* d_n_sym,
                                    uint8_t* d_bits, int64_t bits_cap, int64_t* d_n_bits, void* stream);
/* Host forms (as qpsk_demod_constellation): sym [channels][sym_stride_floats], int64 n_sym[channels] (each in
 * 0..sym_stride_floats/2, else QPSK_ERR_RANGE) -> bits [channels][bits_cap], n_bits[channels]; bits_cap below
 * qpsk_viterbi_bits_bound(max n_sym): QPSK_ERR_CAPACITY with that bound in every n_bits[c] and nothing consumed.
 * Bytes of a row past n_bits[c], up to the longest row of the call, are overwritten. */
QPSK_API int qpsk_viterbi_decode(qpsk_viterbi* p, const float* sym, int64_t sym_stride_floats, const int64_t* n_sym,
                                 uint8_t* bits, int64_t bits_cap, int64_t* n_bits);
QPSK_API int qpsk_viterbi_flush(qpsk_viterbi* p, const float* sym, int64_t sym_stride_floats, const int64_t* n_sym,
                                uint8_t* bits, int64_t bits_cap, int64_t* n_bits);

/* ---- soft-decision frame synchronizer for coded frames ---------------------------------------------------------------- */
/* Not in the reference; it finds coded frames by correlating their known encoded start against the Costas output, so a
 * frame is found when bits of START are wrong, END is not needed, and in coherent mode the Costas lock phase is resolved.
 * Receive path, all on the device (slots = qpsk_fsync_slots_bound(max symbols per call)):
 *   qpsk_demod_constellation_dev -> qpsk_fsync_process_dev -> qpsk_viterbi_flush_dev (a decoder of channels*slots rows,
 *   over the frame rows and d_frame_n_sym) -> qpsk_pack_bits_dev (d_bits + QPSK_CODED_LEAD_BITS + 8*n_start, max_bits =
 *   8*payload_bytes) -> qpsk_rs_decode_dev (d_n_bytes from the synchronizer).
 * Frame format (what modem.coded_frame_bits sends): QPSK_CODED_LEAD_BITS zero bits, START (n_start bytes), payload_bytes
 * bytes, n_end bytes, QPSK_CODED_TAIL_BITS zero bits, MSB first, encoded from state 0 by the K = 7 code above.  One input
 * bit is one symbol, so a frame is F = 32 + 8*(n_start + payload_bytes + n_end) + 6 symbols, and its first P = 32 +
 * 8*n_start symbols are known: the pattern c_0..c_{2P-1}, the code bits of the 32 zeros and START from state 0.
 * Every rule below is exact, and the GPU is bit-identical to tests/fsync_oracle.py.
 * 1. Soft values s0(k), s1(k) of symbol k: rule 1 of the decoder above (same q, forms and scale; differential: symbol k
 *    against symbol k-1).  Positions are absolute symbol indices since create or reset.
 * 2. Correlation at position p, rotation r (the soft values of y*j^-r: r=1 (s1, -s0), r=2 (-s0, -s1), r=3 (-s1, s0)):
 *      M_r(p) = sum_{i<P} (c_{2i} ? 1 : -1) s0_r(p+i) + (c_{2i+1} ? 1 : -1) s1_r(p+i);
 *    coherent: M(p) = max over r = 0..3 (the lowest r on ties); differential: r = 0 only (it is rotation-invariant).
 *    E(p) = sum_{i<P} |s0(p+i)| + |s1(p+i)|.  Integer arithmetic throughout.
 * 3. Detection: the search starts at p = delta (delta = 1 differential, 0 coherent).  Position p is decided once symbols
 *    up to p + 2P - 2 have arrived.  The crossing p0 is the first searched p with E(p) > 0 and 256*M(p) >= rho*E(p); the
 *    frame is at p* = argmax M over [p0, p0 + P) (the lowest p on ties), with rotation r* and metric M(p*), energy
 *    E(p*).  Its window is symbols [p* - delta, p* + F), derotated by j^-r* (an exact swap / negation of I and Q); the
 *    search resumes at p* + F.  A frame goes out in the call after which symbol p* + F - 1 and symbol p0 + 2P - 2 have
 *    both arrived.  qpsk_viterbi_flush_dev on a window (in the handle's mode) emits exactly F bits, and bit i is frame bit i.
 * 4. State per channel (a raw-symbol history of 2P + 1 symbols, the search position, a partial frame of up to F + 1
 *    symbols) lives on the device: any chunking of a stream gives the same frames.
 * rho: 1..256, 0 = QPSK_FSYNC_RHO_DEFAULT (DESIGN.md §3 K15); scale finite and > 0 (the Viterbi defaults fit); n_start
 * 1..24, payload_bytes 1..65536, n_end 0..32; outside: QPSK_ERR_RANGE.  1..16384 channels (else QPSK_ERR_UNSUPPORTED). */
#define QPSK_CODED_LEAD_BITS 32
#define QPSK_CODED_TAIL_BITS 6
#define QPSK_FSYNC_RHO_DEFAULT 144
typedef struct qpsk_fsync qpsk_fsync;
/* one per slot; position -1 and the rest 0 (channel set) in an empty slot */
typedef struct qpsk_fsync_frame {
  int64_t position; /* p* */
  int32_t metric;   /* M(p*) */
  int32_t energy;   /* E(p*) */
  int32_t rotation; /* r*: the window was multiplied by j^-r* */
  int32_t channel;
} qpsk_fsync_frame;
QPSK_API int qpsk_fsync_create(int channels, int differential, float scale, const uint8_t* start_marker, int n_start,
                               int payload_bytes, int n_end, int rho, qpsk_fsync** out);
QPSK_API int qpsk_fsync_destroy(qpsk_fsync* p);
/* back to the state at creation.  Waits for the handle's own stream only. */
QPSK_API int qpsk_fsync_reset(qpsk_fsync* p);
/* P, F, the window length F + delta, and the rho in use */
QPSK_API int qpsk_fsync_shape(const qpsk_fsync* p, int* pattern_syms, int* frame_syms, int* window_syms, int* rho);
/* the most frames one call over at most max_sym symbols per channel completes: ceil(max_sym / F) (frames do not overlap) */
QPSK_API int qpsk_fsync_slots_bound(const qpsk_fsync* p, int64_t max_sym, int64_t* slots);
/* Device: d_sym [channels][sym_stride_floats] cf32 and int d_n_sym[channels] (what qpsk_demod_constellation_dev writes;
 * ragged, 0 allowed; a count past sym_stride_floats/2 is read as sym_stride_floats/2, a negative one as 0) -> per slot
 * c*slots + j, the j-th frame channel c completed in this call: the window in d_frames [channels*slots]
 * [frame_stride_floats] cf32, int d_frame_n_sym (F + delta; 0 for an empty slot; the d_n_sym of qpsk_viterbi_flush_dev),
 * int64 d_n_bytes (payload_bytes; 0 for an empty slot; the count of qpsk_rs_decode_dev) and d_info.  Pointers 8-byte
 * aligned and strides even (else QPSK_ERR_ARG); slots < qpsk_fsync_slots_bound(sym_stride_floats/2) or
 * frame_stride_floats < 2*(F + delta): QPSK_ERR_CAPACITY before anything is enqueued.  Enqueued on `stream` (NULL = the
 * handle's own); the state advances at enqueue, so calls on one handle must run in issue order.  Frame rows of empty
 * slots, and floats of a row past its window, are not written. */
QPSK_API int qpsk_fsync_process_dev(qpsk_fsync* p, const float* d_sym, int64_t sym_stride_floats, const int* d_n_sym,
                                    int slots, float* d_frames, int64_t frame_stride_floats, int* d_frame_n_sym,
                                    int64_t* d_n_bytes, qpsk_fsync_frame* d_info, void* stream);
/* Host form (as qpsk_viterbi_decode): sym [channels][sym_stride_floats], int64 n_sym[channels] (each in
 * 0..sym_stride_floats/2, else QPSK_ERR_RANGE) -> frames [channels*slots][frame_stride_floats], frame_n_sym, n_bytes and
 * info [channels*slots]; slots below qpsk_fsync_slots_bound(max n_sym) or a short frame stride: QPSK_ERR_CAPACITY with
 * that bound in *need_slots and nothing consumed. */
QPSK_API int qpsk_fsync_process(qpsk_fsync* p, const float* sym, int64_t sym_stride_floats, const int64_t* n_sym, int slots,
                                float* frames, int64_t frame_stride_floats, int* frame_n_sym, int64_t* n_bytes,
                                qpsk_fsync_frame* info, int64_t* need_slots);

/* ---- Reed-Solomon outer code over bytes, with byte interleaving -------------------------------------------------------- */
/* Not in the reference; the outer code around the convolutional code (the concatenated scheme): it corrects the short
 * byte bursts the Viterbi decoder leaves.  Receive path, all on the device:
 *   qpsk_demod_constellation_dev -> qpsk_viterbi_flush_dev -> qpsk_demod_frame_bits_dev -> qpsk_rs_decode_dev.
 * The code (fixed at creation; the GPU is bit-identical to tests/rs_oracle.py):
 *   field GF(2^8), primitive polynomial x^8 + x^4 + x^3 + x^2 + 1 (0x11d), alpha = 0x02;
 *   generator g(x) = prod_{j=0}^{nroots-1} (x - alpha^j); nroots even, 2..32, t = nroots/2 symbol errors;
 *   k >= 1 message bytes, n = k + nroots <= 255 (n < 255: a shortened code);
 *   codeword bytes c_0..c_{n-1}, c_0 sent first and the coefficient of x^{n-1}; the message is c_0..c_{k-1} and the parity
 *   c_k..c_{n-1} holds m(x) x^nroots mod g(x) (systematic).
 * Block: depth I (1..8) codewords interleaved byte by byte into I*n bytes; block byte p is byte p / I of codeword p % I.
 * So codeword i carries message bytes i, i+I, i+2I, ..., and the first I*k bytes of a block are its message in order.
 * Decoding rule: a received codeword within Hamming distance t of a codeword of the shortened code becomes that codeword
 * and its status is the distance (0..t); otherwise its status is -1 and its message bytes come out as received.  A
 * correction that would fall in the shortened-away positions is a failure.  The kernels implement the rule exactly with
 * Berlekamp-Massey, Chien search and Forney, accepting a result only when the LFSR length L <= t, deg Lambda = L, Lambda
 * has exactly L distinct roots among the n valid positions, and every Forney magnitude is nonzero (miscorrections of a
 * word more than t from the codeword sent are therefore the same on any implementation of the rule).
 * Statuses are int32, one per codeword, in block order b*I + i.  nroots outside 2..32 or odd, depth outside 1..8:
 * QPSK_ERR_UNSUPPORTED; k < 1 or n > 255: QPSK_ERR_RANGE.
 * The handle holds constants only (generator and tables); calls keep no state, so unlike the other handles its calls may
 * run on any stream, in any order, from any thread. */
typedef struct qpsk_rs qpsk_rs;
QPSK_API int qpsk_rs_create(int nroots, int k, int depth, qpsk_rs** out);
QPSK_API int qpsk_rs_destroy(qpsk_rs* p);
/* host: msg [n_blocks*I*k] -> code [n_blocks*I*n]; decode: code [n_blocks*I*n] -> msg [n_blocks*I*k], status [n_blocks*I] */
QPSK_API int qpsk_rs_encode(qpsk_rs* p, const uint8_t* msg, int64_t n_blocks, uint8_t* code);
QPSK_API int qpsk_rs_decode(qpsk_rs* p, const uint8_t* code, int64_t n_blocks, uint8_t* msg, int* status);
/* device: n_blocks blocks in every row, d_msg [rows][msg_stride] (msg_stride < n_blocks*I*k: QPSK_ERR_ARG) -> d_code
 * [rows][code_stride] (code_stride < n_blocks*I*n: QPSK_ERR_CAPACITY).  Enqueued on `stream` (NULL = the handle's own). */
QPSK_API int qpsk_rs_encode_dev(qpsk_rs* p, const uint8_t* d_msg, int64_t msg_stride, int rows, int64_t n_blocks,
                                uint8_t* d_code, int64_t code_stride, void* stream);
/* device, the rows qpsk_demod_frame_bits_dev / qpsk_demod_bytes_dev write: d_code [rows][code_stride] bytes and int64
 * d_n_bytes[rows], ragged (a count past code_stride is read as code_stride, the framer's "truncated"; a negative one as 0).
 * Each row decodes count / (I*n) whole blocks and ignores a remainder -> d_msg [rows][msg_stride], int64 d_n_msg[rows] =
 * blocks*I*k, int32 d_status [rows][status_stride].  msg_stride < (code_stride / (I*n))*I*k or status_stride <
 * (code_stride / (I*n))*I: QPSK_ERR_CAPACITY before anything is enqueued.  d_n_bytes and d_n_msg 8-byte aligned, d_status
 * 4-byte aligned (else QPSK_ERR_ARG).  Bytes and statuses of a row past what its count gives are not written.  Enqueued
 * on `stream` (NULL = the handle's own). */
QPSK_API int qpsk_rs_decode_dev(qpsk_rs* p, const uint8_t* d_code, int64_t code_stride, const int64_t* d_n_bytes, int rows,
                                uint8_t* d_msg, int64_t msg_stride, int64_t* d_n_msg, int* d_status, int64_t status_stride,
                                void* stream);

/* ---- a6  QPSKModulator  (MS/QPSKModulator.cs:18-168) ---------------------------------------- */
/* tsc_bits: '0'/'1' string or NULL (null/whitespace = no TSC, :27) */
QPSK_API int qpsk_mod_create(int sample_rate, int symbol_rate, double rrc_alpha, int rrc_span,
                             int differential, const char* tsc_bits, qpsk_mod** out);
QPSK_API int qpsk_mod_destroy(qpsk_mod* m);
QPSK_API int qpsk_mod_taps(const qpsk_mod* m, double* out, int cap, int* n);       /* getCoeef() :32 */
/* Modulate(string,bool) :104-167.  out==NULL: size query (*n_floats set).  The modulate calls return
   QPSK_ERR_UNSUPPORTED for sample_rate / symbol_rate > 256 and for more than 96 filter taps per phase
   (ceil(taps / (sample_rate / symbol_rate))); the output is not written then. */
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
/* Opt-in feed-forward AGC stage (qpsk_agc_* above) ahead of everything else: AGC -> FLL? -> MF -> ..., so carriers at any
 * level reach the loops at the level `ref` sets; window 0 = off (the default: the chain is then exactly the reference's).
 * The first W-1 AGC outputs of each channel's stream are discarded once, so the k-th sample reaching the FLL / matched
 * filter is the k-th input sample, scaled (bit alignment as without the stage); the last W-1 samples of a call come out
 * at the start of the next.  The fused symbol-stage kernel and the time-chunk pipeline stay in use with the stage on.
 * May be called at any time: synchronises the handle, resets this stage only (history, discard count).  Limits and
 * argument codes as qpsk_agc_create_batch. */
QPSK_API int qpsk_demod_set_agc(qpsk_demod* d, int window, float ref, float max_gain);
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
/* qpsk_demod_frame_bits on DEVICE bits: d_bits [channels][bits_stride], one byte 0/1 per bit, int64 d_n_bits[channels]
 * (each in 0..bits_stride: device memory, not checked) -> d_payload [channels][payload_cap], d_n_bytes[channels] as
 * qpsk_demod_bytes_dev.  Shares the framer state with the other framer calls.  With qpsk_viterbi_decode_dev it keeps the
 * coded receive path on the device.  Enqueued on `stream` (NULL = the handle's own), no synchronisation. */
QPSK_API int qpsk_demod_frame_bits_dev(qpsk_demod* d, const uint8_t* d_bits, int64_t bits_stride, const int64_t* d_n_bits,
                                       const uint8_t* start_marker, int64_t n_start, const uint8_t* end_marker, int64_t n_end,
                                       uint8_t* d_payload, int64_t payload_cap, int64_t* d_n_bytes, void* stream);
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
