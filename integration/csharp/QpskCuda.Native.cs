// integration/csharp/QpskCuda.Native.cs -> Modulation-Simulation/Native/QpskCuda.cs (new file)
// P/Invoke surface of libqpskcuda.so (include/qpskcuda.h).  Not built in this repository: the image has no .NET toolchain.
using System;
using System.Runtime.InteropServices;

namespace QPSK.Native;

internal static unsafe partial class QpskCuda
{
    const string Lib = "qpskcuda";   // libqpskcuda.so / qpskcuda.dll next to the assembly

    // status -> the exception the managed code used to throw at the same place
    internal static void Check(int st, string? arg = null)
    {
        switch (st)
        {
            case 0: return;
            case -1: throw new ArgumentNullException(arg);
            case -2: throw new ArgumentException(Marshal.PtrToStringAnsi(qpsk_strerror(st)), arg);
            case -3: throw new ArgumentOutOfRangeException(arg);
            default:
                throw new InvalidOperationException(
                    $"qpskcuda status {st}: {Marshal.PtrToStringAnsi(qpsk_strerror(st))} " +
                    Marshal.PtrToStringAnsi(qpsk_last_cuda_error()));
        }
    }

    [DllImport(Lib)] internal static extern IntPtr qpsk_strerror(int status);
    [DllImport(Lib)] internal static extern IntPtr qpsk_last_cuda_error();
    [DllImport(Lib)] internal static extern int qpsk_set_device(int ordinal);

    // a1  RRCFilter.generateCoefficents            (MS/Models/RRC-filter.cs:16)
    [DllImport(Lib)] internal static extern int qpsk_rrc_taps(double span, double beta, int fs, int rs,
                                                              double* outTaps, int cap, out int n);
    // a2-a5  ComplexFIRFilter                       (MS/Models/FIRFilter.cs:29,80,96)
    [DllImport(Lib)] internal static extern int qpsk_fir_create(float* tapsIq, int nFloats, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_fir_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_fir_filter(IntPtr h, float* iqIn, float* iqOut, long nFloats, long outCap);
    [DllImport(Lib)] internal static extern int qpsk_fir_fft_filter(IntPtr h, float* iqIn, float* iqOut, long nFloats);
    [DllImport(Lib)] internal static extern int qpsk_fir_set_mode(IntPtr h, int mode);   // QPSK_FIR_FAST 0 / EXACT 1 / FMA 2 / SPLIT 3
    // a7-a8  FLLBandEdgeFilter                      (MS/Models/Band-Edge Filter.cs:40,64)
    [DllImport(Lib)] internal static extern int qpsk_fll_create(float sps, float rolloff, int filterSize, float bw, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_fll_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_fll_process(IntPtr h, float* iqIn, float* iqOut, long nFloats, long outCap);
    [DllImport(Lib)] internal static extern int qpsk_fll_get_state(IntPtr h, out float phase, out float freq);
    [DllImport(Lib)] internal static extern int qpsk_fll_set_state(IntPtr h, in float phase, in float freq);
    // a9  MuellerMuller                             (MS/Models/MuellerMuller.cs:38,52)
    [DllImport(Lib)] internal static extern int qpsk_mm_create(double sps, double kp, double ki, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_mm_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_mm_process(IntPtr h, float* mfIn, long nFloats, float* symOut, long capFloats, out int nSym);
    // a10  CostasLoopQpsk                           (MS/Models/CostasLoopQpsk.cs:29,98,130)
    [DllImport(Lib)] internal static extern int qpsk_costas_create(double fs, double bwHz, double damping, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_costas_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_costas_process(IntPtr h, float* iqIn, float* iqOut, long nFloats, long outCap);
    [DllImport(Lib)] internal static extern int qpsk_costas_get_state(IntPtr h, out double theta, out double freq);
    // symbol-spaced blind CMA equalizer              (not in the reference; spec in include/qpskcuda.h)
    [DllImport(Lib)] internal static extern int qpsk_eq_create(int nTaps, float mu, float modulus, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_eq_create_fractional(int nTaps, float mu, float modulus, int sps, int channels, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_eq_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_eq_reset(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_eq_process(IntPtr h, float* iqIn, float* iqOut, long nFloats, long outCap);
    [DllImport(Lib)] internal static extern int qpsk_eq_get_taps(IntPtr h, float* tapsIq, long capFloats);
    [DllImport(Lib)] internal static extern int qpsk_eq_set_taps(IntPtr h, float* tapsIq, long nFloats);
    [DllImport(Lib)] internal static extern int qpsk_pfb_taps(int channels, int tapsPerBranch, double cutoff, double attenDb, double* taps, int cap, out int n);
    [DllImport(Lib)] internal static extern int qpsk_pfb_create(float* taps, int nTaps, int channels, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_pfb_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_pfb_reset(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_pfb_process(IntPtr h, float* iqIn, long nFloats, float* iqOut, long outStrideFloats, out long nOutFloats);
    [DllImport(Lib)] internal static extern int qpsk_pfb_process_dev(IntPtr h, float* dIn, long nFloats, float* dOut, long outStrideFloats, out long nOutFloats, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_ddc_create(float* taps, int nTaps, double* freqs, int channels, int decim, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_ddc_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_ddc_reset(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_ddc_process(IntPtr h, float* iqIn, long nFloats, float* iqOut, long outStrideFloats, out long nOutFloats);
    [DllImport(Lib)] internal static extern int qpsk_ddc_process_dev(IntPtr h, float* dIn, long nFloats, float* dOut, long outStrideFloats, out long nOutFloats, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_agc_create_batch(int window, float refLevel, float maxGain, int channels, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_agc_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_agc_reset(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_agc_process(IntPtr h, float* iqIn, float* iqOut, long nFloats, long outCapFloats);
    [DllImport(Lib)] internal static extern int qpsk_agc_process_dev(IntPtr h, float* dIn, float* dOut, long nFloats, long inStrideFloats, long outStrideFloats, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_agc_gain(IntPtr h, float* gain, long cap);
    [DllImport(Lib)] internal static extern int qpsk_agc_gain_dev(IntPtr h, float* dGain, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_resamp_create(float* taps, int nTaps, int interp, int decim, int channels, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_resamp_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_resamp_reset(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_resamp_process(IntPtr h, float* iqIn, long nFloats, float* iqOut, long outStrideFloats, out long nOutFloats);
    [DllImport(Lib)] internal static extern int qpsk_resamp_process_dev(IntPtr h, float* dIn, long nFloats, long inStrideFloats, float* dOut, long outStrideFloats, out long nOutFloats, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_conv_create(int channels, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_conv_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_conv_reset(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_conv_encode(IntPtr h, byte* bits, long nBits, byte* output);
    [DllImport(Lib)] internal static extern int qpsk_conv_encode_dev(IntPtr h, byte* dBits, long nBits, long bitsStride, byte* dOut, long outStride, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_viterbi_create(int channels, int differential, float scale, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_viterbi_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_viterbi_reset(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_viterbi_bits_bound(IntPtr h, long maxSym, out long cap);
    [DllImport(Lib)] internal static extern int qpsk_viterbi_decode_dev(IntPtr h, float* dSym, long symStrideFloats, int* dNSym, byte* dBits, long bitsCap, long* dNBits, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_viterbi_flush_dev(IntPtr h, float* dSym, long symStrideFloats, int* dNSym, byte* dBits, long bitsCap, long* dNBits, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_viterbi_decode(IntPtr h, float* sym, long symStrideFloats, long* nSym, byte* bits, long bitsCap, long* nBits);
    [DllImport(Lib)] internal static extern int qpsk_viterbi_flush(IntPtr h, float* sym, long symStrideFloats, long* nSym, byte* bits, long bitsCap, long* nBits);
    [DllImport(Lib)] internal static extern int qpsk_fsync_create(int channels, int differential, float scale, byte* startMarker, int nStart, int payloadBytes, int nEnd, int rho, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_fsync_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_fsync_reset(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_fsync_shape(IntPtr h, out int patternSyms, out int frameSyms, out int windowSyms, out int rho);
    [DllImport(Lib)] internal static extern int qpsk_fsync_slots_bound(IntPtr h, long maxSym, out long slots);
    [DllImport(Lib)] internal static extern int qpsk_fsync_process_dev(IntPtr h, float* dSym, long symStrideFloats, int* dNSym, int slots, float* dFrames, long frameStrideFloats, int* dFrameNSym, long* dNBytes, IntPtr dInfo, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_fsync_process(IntPtr h, float* sym, long symStrideFloats, long* nSym, int slots, float* frames, long frameStrideFloats, int* frameNSym, long* nBytes, IntPtr info, out long needSlots);
    [DllImport(Lib)] internal static extern int qpsk_rs_create(int nroots, int k, int depth, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_rs_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_rs_encode(IntPtr h, byte* msg, long nBlocks, byte* code);
    [DllImport(Lib)] internal static extern int qpsk_rs_decode(IntPtr h, byte* code, long nBlocks, byte* msg, int* status);
    [DllImport(Lib)] internal static extern int qpsk_rs_encode_dev(IntPtr h, byte* dMsg, long msgStride, int rows, long nBlocks, byte* dCode, long codeStride, IntPtr stream);
    [DllImport(Lib)] internal static extern int qpsk_rs_decode_dev(IntPtr h, byte* dCode, long codeStride, long* dNBytes, int rows, byte* dMsg, long msgStride, long* dNMsg, int* dStatus, long statusStride, IntPtr stream);
    // a6  QPSKModulator                             (MS/QPSKModulator.cs:18,54,104)
    [DllImport(Lib, CharSet = CharSet.Ansi)]
    internal static extern int qpsk_mod_create(int fs, int rs, double alpha, int span, int diff, string? tsc, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_mod_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_mod_taps(IntPtr h, double* outTaps, int cap, out int n);
    [DllImport(Lib)] internal static extern int qpsk_mod_modulate_bits(IntPtr h, byte* bits, long nBits, int pulse, float* iqOut, long capFloats, out long nFloats);
    [DllImport(Lib)] internal static extern int qpsk_mod_modulate_bytes(IntPtr h, byte* payload, long nPayload, byte* start, long nStart,
                                                                        byte* end, long nEnd, int pulse, float* iqOut, long capFloats, out long nFloats);
    // a11-a12  QPSKDeModulator                      (MS/QPSKDeModulator.cs:11,169,345,427)
    [DllImport(Lib, CharSet = CharSet.Ansi)]
    internal static extern int qpsk_demod_create(int fs, int rs, float alpha, int span, double symBw, double costasBw, double cfoBw,
                                                 int diff, string? tsc, int useFll, long maxFrameBytes, out IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_demod_destroy(IntPtr h);
    [DllImport(Lib)] internal static extern int qpsk_demod_set_equalizer(IntPtr h, int nTaps, float mu, float modulus);
    [DllImport(Lib)] internal static extern int qpsk_demod_equalizer_taps(IntPtr h, float* tapsIq, long capFloats);
    [DllImport(Lib)] internal static extern int qpsk_demod_set_fractional_equalizer(IntPtr h, int nTaps, float mu, float modulus);
    [DllImport(Lib)] internal static extern int qpsk_demod_set_agc(IntPtr h, int window, float refLevel, float maxGain);
    [DllImport(Lib)] internal static extern int qpsk_demod_fractional_equalizer_taps(IntPtr h, float* tapsIq, long capFloats);
    [DllImport(Lib)] internal static extern int qpsk_demod_bits(IntPtr h, float* iqIn, long nFloats, byte* bitsOut, long cap, out long nBits);
    [DllImport(Lib)] internal static extern int qpsk_demod_bytes(IntPtr h, float* iqIn, long nFloats, byte* start, long nStart,
                                                                 byte* end, long nEnd, byte* payloadOut, long cap, out long nBytes);
    [DllImport(Lib)] internal static extern int qpsk_demod_last_payload(IntPtr h, byte* payloadOut, long cap, out long nBytes);
    [DllImport(Lib)] internal static extern int qpsk_demod_constellation(IntPtr h, float* iqIn, long nFloats, float* symOut, long capFloats, out long nSym);
    [DllImport(Lib)] internal static extern int qpsk_demod_frame_bits(IntPtr h, byte* bits01, long bitsStride, long* nBits, byte* start, long nStart,
                                                                      byte* end, long nEnd, byte* payloadOut, long cap, long* nBytes);
}
