// integration/csharp/QpskCuda.Shim.cs — the reference's public classes on the hot path with their bodies replaced by
// calls into libqpskcuda.so.  Same namespaces, class names, constructor and method signatures, defaults, RETURN VALUES and
// exceptions as Modulation-Simulation/{Models/FIRFilter.cs, Models/RRC-filter.cs, Models/Band-Edge Filter.cs,
// Models/MuellerMuller.cs, Models/CostasLoopQpsk.cs, QPSKModulator.cs, QPSKDeModulator.cs}; each member cites the line it
// stands in for.  The managed argument checks of the reference run BEFORE the native call, in the reference's order, so a
// caller sees the same exception type and parameter name.  Loop and filter state lives on the device inside the native
// handle, one handle per object, exactly as the managed objects were one per stream.  HelperFunctions (BitPacker,
// SaveAsCs16, ...) and RealFIRFilter stay as they are.
// Not built in this repository: the image has no .NET toolchain.  tests/test_cabi_cpu.py checks every binding against the
// header and every Process() return expression against the reference's convention.
using System;
using System.Runtime.InteropServices;
using System.Text;
using QPSK.Native;

namespace QPSK.Native
{
    // Owns one native handle.  The reference classes are not IDisposable and existing callers never dispose them, so the
    // device buffers and CUDA streams behind a handle are released by the SafeHandle's critical finaliser once the managed
    // object is unreachable; Dispose() on the shim classes is an optional early release.
    internal sealed class QpskHandle : SafeHandle
    {
        readonly Func<IntPtr, int> _destroy;
        public QpskHandle(IntPtr h, Func<IntPtr, int> destroy) : base(IntPtr.Zero, true) { _destroy = destroy; SetHandle(h); }
        public override bool IsInvalid => handle == IntPtr.Zero;
        protected override bool ReleaseHandle() => _destroy(handle) == 0;
        public IntPtr Ptr => (IsClosed || IsInvalid) ? throw new ObjectDisposedException(nameof(QpskHandle)) : handle;
    }
}

namespace QPSK.Models
{
    public class RRCFilter
    {
        public static unsafe double[] generateCoefficents(double spanSymbols, double beta, int sampleRate, int SymbolRate)   // RRC-filter.cs:16
        {
            QpskCuda.Check(QpskCuda.qpsk_rrc_taps(spanSymbols, beta, sampleRate, SymbolRate, null, 0, out int n));
            var h = new double[n];
            fixed (double* p = h) QpskCuda.Check(QpskCuda.qpsk_rrc_taps(spanSymbols, beta, sampleRate, SymbolRate, p, n, out n));
            return h;
        }
    }

    public sealed unsafe class ComplexFIRFilter : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly float[] taps;                                                // FIRFilter.cs:11
        public ComplexFIRFilter(float[] tapsInterleavedIQ)                         // :29
        {
            if (tapsInterleavedIQ == null) throw new ArgumentNullException(nameof(tapsInterleavedIQ));                                        // :31
            if ((tapsInterleavedIQ.Length & 1) != 0) throw new ArgumentException("Taps must be interleaved IQ with even length.", nameof(tapsInterleavedIQ));   // :32
            if (tapsInterleavedIQ.Length == 0) throw new ArgumentException("Taps cannot be empty.", nameof(tapsInterleavedIQ));               // :33
            taps = (float[])tapsInterleavedIQ.Clone();
            IntPtr h;
            fixed (float* t = tapsInterleavedIQ)
                QpskCuda.Check(QpskCuda.qpsk_fir_create(t, tapsInterleavedIQ.Length, out h), nameof(tapsInterleavedIQ));
            _o = new QpskHandle(h, QpskCuda.qpsk_fir_destroy);
        }
        public void Filter(float inI, float inQ, out float outI, out float outQ)   // :59  one sample = a 2-float span
        {
            float* io = stackalloc float[4];
            io[0] = inI; io[1] = inQ;
            QpskCuda.Check(QpskCuda.qpsk_fir_filter(_h, io, io + 2, 2, 2));
            outI = io[2]; outQ = io[3];
            GC.KeepAlive(this);
        }
        public void Filter(ReadOnlySpan<float> iqIn, Span<float> iqOut)            // :80  streaming, delay line on the device
        {
            if ((iqIn.Length & 1) != 0) throw new ArgumentException("Input must be interleaved IQ with even length.", nameof(iqIn));   // :82
            if (iqOut.Length < iqIn.Length) throw new ArgumentException("Output span is too small.", nameof(iqOut));                  // :83
            fixed (float* i = iqIn) fixed (float* o = iqOut)
                QpskCuda.Check(QpskCuda.qpsk_fir_filter(_h, i, o, iqIn.Length, iqOut.Length), nameof(iqIn));
            GC.KeepAlive(this);
        }
        public float[] fftFilter(float[] iqData)                                   // :96  stateless, offset N-1
        {
            if (iqData == null) throw new ArgumentNullException(nameof(iqData));                                                       // :98
            if ((iqData.Length & 1) != 0) throw new ArgumentException("Data must be interleaved IQ with even length.", nameof(iqData));   // :99
            if (iqData.Length == 0) return Array.Empty<float>();                                                                      // :100
            var y = new float[iqData.Length];
            fixed (float* i = iqData) fixed (float* o = y)
                QpskCuda.Check(QpskCuda.qpsk_fir_fft_filter(_h, i, o, iqData.Length), nameof(iqData));
            GC.KeepAlive(this);
            return y;
        }
        /// <summary>Not in the reference: result mode of this handle (include/qpskcuda.h QPSK_FIR_*).  Fast = fp32 FMA, kernel picked
        /// by the library (within 1e-5 of the reference); Exact = the reference's summation order, bit for bit; Fma / Split pin
        /// one of the two FMA kernels.</summary>
        public enum Mode { Fast = 0, Exact = 1, Fma = 2, Split = 3 }
        public void SetMode(Mode mode)
        {
            QpskCuda.Check(QpskCuda.qpsk_fir_set_mode(_h, (int)mode), nameof(mode));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    public sealed unsafe class FLLBandEdgeFilter : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public float sps, rolloff, bandwidth;                                        // Band-Edge Filter.cs:19-22
        public int filterSize;
        public float phase                                                           // :25 (a public field upstream)
        {
            get { QpskCuda.Check(QpskCuda.qpsk_fll_get_state(_h, out float p, out _)); GC.KeepAlive(this); return p; }
            set { QpskCuda.Check(QpskCuda.qpsk_fll_get_state(_h, out _, out float f)); QpskCuda.Check(QpskCuda.qpsk_fll_set_state(_h, in value, in f)); GC.KeepAlive(this); }
        }
        public float freq                                                            // :26
        {
            get { QpskCuda.Check(QpskCuda.qpsk_fll_get_state(_h, out _, out float f)); GC.KeepAlive(this); return f; }
            set { QpskCuda.Check(QpskCuda.qpsk_fll_get_state(_h, out float p, out _)); QpskCuda.Check(QpskCuda.qpsk_fll_set_state(_h, in p, in value)); GC.KeepAlive(this); }
        }
        public FLLBandEdgeFilter(float sps, float rolloff, int filterSize, float bandwidth)   // :40 (range checks :42-45 -> status -3)
        {
            this.sps = sps; this.rolloff = rolloff; this.filterSize = filterSize; this.bandwidth = bandwidth;
            QpskCuda.Check(QpskCuda.qpsk_fll_create(sps, rolloff, filterSize, bandwidth, out IntPtr h));
            _o = new QpskHandle(h, QpskCuda.qpsk_fll_destroy);
        }
        public int Process(ReadOnlySpan<float> inputIQ, Span<float> outputIQ)       // :64
        {
            if ((inputIQ.Length & 1) != 0) throw new ArgumentException("Input must be interleaved IQ with even length.", nameof(inputIQ));   // :66
            if (outputIQ.Length < inputIQ.Length) throw new ArgumentException("Output span is too small.", nameof(outputIQ));              // :68
            fixed (float* i = inputIQ) fixed (float* o = outputIQ)
                QpskCuda.Check(QpskCuda.qpsk_fll_process(_h, i, o, inputIQ.Length, outputIQ.Length), nameof(inputIQ));
            GC.KeepAlive(this);
            return inputIQ.Length >> 1;                                              // complex samples processed (:71, :86)
        }
        public float[] Process(float[] inputIQ)                                      // :90
        {
            if (inputIQ == null) throw new ArgumentNullException(nameof(inputIQ));
            var y = new float[inputIQ.Length];
            Process(inputIQ.AsSpan(), y.AsSpan());
            return y;
        }
        public void Process(float inI, float inQ, out float outI, out float outQ)   // :102
        {
            float* io = stackalloc float[4];
            io[0] = inI; io[1] = inQ;
            QpskCuda.Check(QpskCuda.qpsk_fll_process(_h, io, io + 2, 2, 2));
            outI = io[2]; outQ = io[3];
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    public sealed unsafe class MuellerMuller : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public MuellerMuller(double samplesPerSymbol, double kp, double ki)          // MuellerMuller.cs:38
        {
            QpskCuda.Check(QpskCuda.qpsk_mm_create(samplesPerSymbol, kp, ki, out IntPtr h));
            _o = new QpskHandle(h, QpskCuda.qpsk_mm_destroy);
        }
        public int Process(ReadOnlySpan<float> incomingMfSamplesIQ, Span<float> outputSymbolsIQ)   // :52
        {
            if ((incomingMfSamplesIQ.Length & 1) != 0)
                throw new ArgumentException("Input must be interleaved IQ with even length.", nameof(incomingMfSamplesIQ));   // :54-55
            int nSym;
            fixed (float* i = incomingMfSamplesIQ) fixed (float* o = outputSymbolsIQ)
                QpskCuda.Check(QpskCuda.qpsk_mm_process(_h, i, incomingMfSamplesIQ.Length, o, outputSymbolsIQ.Length, out nSym),
                               nameof(incomingMfSamplesIQ));
            GC.KeepAlive(this);
            return nSym;          // outSymbols: complex symbols written (:135); QPSKDeModulator.cs:364-375 loops k < nSymbols over it
        }
        public float[] Process(float[] incomingMfSamplesIQ)                          // :141
        {
            if (incomingMfSamplesIQ == null) throw new ArgumentNullException(nameof(incomingMfSamplesIQ));
            if ((incomingMfSamplesIQ.Length & 1) != 0)
                throw new ArgumentException("Input must be interleaved IQ with even length.", nameof(incomingMfSamplesIQ));
            int maxSymbols = incomingMfSamplesIQ.Length >> 1;                        // :148
            var tmp = new float[maxSymbols << 1];                                    // :149
            int n = Process(incomingMfSamplesIQ.AsSpan(), tmp.AsSpan());             // :151
            if (n == maxSymbols) return tmp;                                         // :152
            var y = new float[n << 1];                                               // :154
            Array.Copy(tmp, y, y.Length);
            return y;
        }
        public void Dispose() => _o.Dispose();
    }

    public sealed unsafe class CostasLoopQpsk : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public CostasLoopQpsk(double sampleRate, double loopBandwidthHz, double damping = 0.707)   // CostasLoopQpsk.cs:29
        {
            QpskCuda.Check(QpskCuda.qpsk_costas_create(sampleRate, loopBandwidthHz, damping, out IntPtr h));
            _o = new QpskHandle(h, QpskCuda.qpsk_costas_destroy);
        }
        public static void GetSign(float i, float q, out float di, out float dq)    // :52 (pure host helper, unchanged)
        {
            di = (i >= 0f) ? 1f : -1f;
            dq = (q >= 0f) ? 1f : -1f;
        }
        public void Process(float inI, float inQ, out float outI, out float outQ)   // :63
        {
            float* io = stackalloc float[4];
            io[0] = inI; io[1] = inQ;
            QpskCuda.Check(QpskCuda.qpsk_costas_process(_h, io, io + 2, 2, 2));
            outI = io[2]; outQ = io[3];
            GC.KeepAlive(this);
        }
        public int Process(ReadOnlySpan<float> iqIn, Span<float> iqOut)             // :98
        {
            if ((iqIn.Length & 1) != 0) throw new ArgumentException("Input must be interleaved IQ with even length.", nameof(iqIn));   // :100
            if (iqOut.Length < iqIn.Length) throw new ArgumentException("Output span is too small.", nameof(iqOut));                  // :102
            fixed (float* i = iqIn) fixed (float* o = iqOut)
                QpskCuda.Check(QpskCuda.qpsk_costas_process(_h, i, o, iqIn.Length, iqOut.Length), nameof(iqIn));
            GC.KeepAlive(this);
            return iqIn.Length >> 1;                                                 // complex samples processed (:105, :113)
        }
        public float[] Process(float[] iqIn)                                         // :119
        {
            if (iqIn == null) throw new ArgumentNullException(nameof(iqIn));
            var y = new float[iqIn.Length];
            Process(iqIn.AsSpan(), y.AsSpan());
            return y;
        }
        public (double theta, double freq) GetState()                                // :130
        {
            QpskCuda.Check(QpskCuda.qpsk_costas_get_state(_h, out double t, out double f));
            GC.KeepAlive(this);
            return (t, f);
        }
        public void Dispose() => _o.Dispose();
    }

    // Blind CMA equalizer: not a reference class (its receive chain has none); the block a GNU Radio PSK receiver puts
    // between clock recovery and the Costas loop, or (sps 2..8) fractionally spaced ahead of it.  Arithmetic spec in
    // include/qpskcuda.h.
    public sealed unsafe class CmaEqualizer : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int NumTaps;
        public CmaEqualizer(int nTaps, float mu, float modulus = 1.0f)
        {
            QpskCuda.Check(QpskCuda.qpsk_eq_create(nTaps, mu, modulus, out IntPtr h));
            _o = new QpskHandle(h, QpskCuda.qpsk_eq_destroy);
            NumTaps = nTaps;
        }
        // fractionally spaced: input at sps samples per symbol, the taps update on every sps-th sample (sps 1..8)
        public CmaEqualizer(int nTaps, float mu, float modulus, int sps)
        {
            QpskCuda.Check(QpskCuda.qpsk_eq_create_fractional(nTaps, mu, modulus, sps, 1, out IntPtr h));
            _o = new QpskHandle(h, QpskCuda.qpsk_eq_destroy);
            NumTaps = nTaps;
        }
        public int Process(ReadOnlySpan<float> iqIn, Span<float> iqOut)
        {
            if ((iqIn.Length & 1) != 0) throw new ArgumentException("Input must be interleaved IQ with even length.", nameof(iqIn));
            if (iqOut.Length < iqIn.Length) throw new ArgumentException("Output span is too small.", nameof(iqOut));
            fixed (float* i = iqIn) fixed (float* o = iqOut)
                QpskCuda.Check(QpskCuda.qpsk_eq_process(_h, i, o, iqIn.Length, iqOut.Length), nameof(iqIn));
            GC.KeepAlive(this);
            return iqIn.Length >> 1;                                                 // complex symbols processed
        }
        public float[] Process(float[] iqIn)
        {
            if (iqIn == null) throw new ArgumentNullException(nameof(iqIn));
            var y = new float[iqIn.Length];
            Process(iqIn.AsSpan(), y.AsSpan());
            return y;
        }
        public float[] Taps                                                          // interleaved IQ, 2 * NumTaps floats
        {
            get
            {
                var t = new float[2 * NumTaps];
                fixed (float* p = t) QpskCuda.Check(QpskCuda.qpsk_eq_get_taps(_h, p, t.Length));
                GC.KeepAlive(this);
                return t;
            }
            set
            {
                if (value == null) throw new ArgumentNullException(nameof(value));
                fixed (float* p = value) QpskCuda.Check(QpskCuda.qpsk_eq_set_taps(_h, p, value.Length), nameof(value));
                GC.KeepAlive(this);
            }
        }
        public void Reset()
        {
            QpskCuda.Check(QpskCuda.qpsk_eq_reset(_h));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    // Polyphase analysis channelizer (not in the reference): one wideband stream -> Channels streams at 1/Channels of the
    // rate, channel k centred at +k/Channels cycles per input sample; rows [Channels][outStride] are what the batch
    // QPSKDeModulator reads.  State persists across calls.
    public sealed unsafe class PfbChannelizer : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int Channels;
        public PfbChannelizer(float[] taps, int channels)
        {
            if (taps == null) throw new ArgumentNullException(nameof(taps));
            if (taps.Length == 0) throw new ArgumentException("Prototype taps must not be empty.", nameof(taps));
            if (channels < 2 || channels > 1024 || (channels & (channels - 1)) != 0)
                throw new ArgumentOutOfRangeException(nameof(channels), "channels must be a power of two from 2 to 1024.");
            IntPtr h;
            fixed (float* t = taps) QpskCuda.Check(QpskCuda.qpsk_pfb_create(t, taps.Length, channels, out h), nameof(taps));
            _o = new QpskHandle(h, QpskCuda.qpsk_pfb_destroy);
            Channels = channels;
        }
        // Kaiser-windowed sinc prototype, unit DC gain, channels * tapsPerBranch taps; cutoff in cycles per input sample
        public static double[] DesignTaps(int channels, int tapsPerBranch, double cutoff, double attenDb = 60.0)
        {
            QpskCuda.Check(QpskCuda.qpsk_pfb_taps(channels, tapsPerBranch, cutoff, attenDb, null, 0, out int n));
            var t = new double[n];
            fixed (double* p = t) QpskCuda.Check(QpskCuda.qpsk_pfb_taps(channels, tapsPerBranch, cutoff, attenDb, p, n, out n));
            return t;
        }
        // iqIn: interleaved IQ of the wideband stream; iqOut: [Channels][outStrideFloats].  Returns floats written per channel.
        public long Process(ReadOnlySpan<float> iqIn, Span<float> iqOut, long outStrideFloats)
        {
            if ((iqIn.Length & 1) != 0) throw new ArgumentException("Input must be interleaved IQ with even length.", nameof(iqIn));
            if (outStrideFloats < 0 || iqOut.Length < Channels * outStrideFloats)
                throw new ArgumentException("Output span is too small for Channels rows of outStrideFloats.", nameof(iqOut));
            long n;
            fixed (float* i = iqIn) fixed (float* o = iqOut)
                QpskCuda.Check(QpskCuda.qpsk_pfb_process(_h, i, iqIn.Length, o, outStrideFloats, out n), nameof(iqOut));
            GC.KeepAlive(this);
            return n;
        }
        public void Reset()
        {
            QpskCuda.Check(QpskCuda.qpsk_pfb_reset(_h));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    // Digital down-converter bank (not in the reference): one wideband stream -> one channel per frequency (cycles per
    // input sample, in [-0.5, 0.5)), each mixed down, lowpass-filtered with the shared real prototype and decimated by
    // Decim; rows [Channels][outStride] are what the batch QPSKDeModulator reads.  State persists across calls.
    public sealed unsafe class DdcBank : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int Channels;
        public readonly int Decim;
        public DdcBank(float[] taps, double[] freqs, int decim)
        {
            if (taps == null) throw new ArgumentNullException(nameof(taps));
            if (freqs == null) throw new ArgumentNullException(nameof(freqs));
            if (taps.Length == 0) throw new ArgumentException("Prototype taps must not be empty.", nameof(taps));
            if (taps.Length > 4096) throw new ArgumentOutOfRangeException(nameof(taps), "At most 4096 prototype taps.");
            if (freqs.Length < 1 || freqs.Length > 2048)
                throw new ArgumentOutOfRangeException(nameof(freqs), "From 1 to 2048 channel frequencies.");
            if (decim < 1 || decim > 1024) throw new ArgumentOutOfRangeException(nameof(decim), "decim must be from 1 to 1024.");
            foreach (var f in freqs)
                if (!(f >= -0.5 && f < 0.5))
                    throw new ArgumentOutOfRangeException(nameof(freqs), "Frequencies are cycles per input sample in [-0.5, 0.5).");
            IntPtr h;
            fixed (float* t = taps) fixed (double* f = freqs)
                QpskCuda.Check(QpskCuda.qpsk_ddc_create(t, taps.Length, f, freqs.Length, decim, out h), nameof(taps));
            _o = new QpskHandle(h, QpskCuda.qpsk_ddc_destroy);
            Channels = freqs.Length;
            Decim = decim;
        }
        // iqIn: interleaved IQ of the wideband stream; iqOut: [Channels][outStrideFloats].  Returns floats written per channel.
        public long Process(ReadOnlySpan<float> iqIn, Span<float> iqOut, long outStrideFloats)
        {
            if ((iqIn.Length & 1) != 0) throw new ArgumentException("Input must be interleaved IQ with even length.", nameof(iqIn));
            if (outStrideFloats < 0 || iqOut.Length < Channels * outStrideFloats)
                throw new ArgumentException("Output span is too small for Channels rows of outStrideFloats.", nameof(iqOut));
            long n;
            fixed (float* i = iqIn) fixed (float* o = iqOut)
                QpskCuda.Check(QpskCuda.qpsk_ddc_process(_h, i, iqIn.Length, o, outStrideFloats, out n), nameof(iqOut));
            GC.KeepAlive(this);
            return n;
        }
        public void Reset()
        {
            QpskCuda.Check(QpskCuda.qpsk_ddc_reset(_h));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    // Feed-forward AGC (not in the reference; definition in qpskcuda.h): per channel every sample is scaled by
    // min(refLevel / m, maxGain), m the peak of max(|I|, |Q|) over a Window-sample window looking Window-1 samples ahead, so
    // the output is the input delayed by Window-1 samples, at level refLevel.  State persists across calls.
    public sealed unsafe class Agc : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int Window;
        public readonly int Channels;
        public Agc(int window, float refLevel = 1.0f, float maxGain = 65536.0f, int channels = 1)
        {
            if (window < 1 || window > 4096) throw new ArgumentOutOfRangeException(nameof(window), "window must be from 1 to 4096.");
            if (!(refLevel > 0) || float.IsInfinity(refLevel)) throw new ArgumentOutOfRangeException(nameof(refLevel), "refLevel must be finite and > 0.");
            if (!(maxGain > 0) || float.IsInfinity(maxGain)) throw new ArgumentOutOfRangeException(nameof(maxGain), "maxGain must be finite and > 0.");
            if (channels < 1) throw new ArgumentOutOfRangeException(nameof(channels), "At least one channel.");
            IntPtr h;
            QpskCuda.Check(QpskCuda.qpsk_agc_create_batch(window, refLevel, maxGain, channels, out h), nameof(window));
            _o = new QpskHandle(h, QpskCuda.qpsk_agc_destroy);
            Window = window;
            Channels = channels;
        }
        // iqIn / iqOut: [Channels][nFloats] interleaved IQ, nFloats = iqIn.Length / Channels.
        public void Process(ReadOnlySpan<float> iqIn, Span<float> iqOut)
        {
            if (iqIn.Length % (2 * Channels) != 0)
                throw new ArgumentException("Input must be Channels rows of interleaved IQ with even length.", nameof(iqIn));
            if (iqOut.Length < iqIn.Length) throw new ArgumentException("Output span is shorter than the input.", nameof(iqOut));
            long n = iqIn.Length / Channels;
            fixed (float* i = iqIn) fixed (float* o = iqOut)
                QpskCuda.Check(QpskCuda.qpsk_agc_process(_h, i, o, n, n), nameof(iqOut));
            GC.KeepAlive(this);
        }
        // the gain of each channel's last output
        public float[] Gain()
        {
            var g = new float[Channels];
            fixed (float* p = g) QpskCuda.Check(QpskCuda.qpsk_agc_gain(_h, p, g.Length));
            GC.KeepAlive(this);
            return g;
        }
        public void Reset()
        {
            QpskCuda.Check(QpskCuda.qpsk_agc_reset(_h));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    // Rational resampler (not in the reference; definition in qpskcuda.h): Channels streams, each interpolated by Interp,
    // filtered with a real prototype and decimated by Decim (scipy.signal.upfirdn per channel, streamed).  No Interp factor:
    // taps summing to Interp pass a carrier with unit gain.  State persists across calls: any chunking gives the same outputs.
    public sealed unsafe class Resampler : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int Interp;
        public readonly int Decim;
        public readonly int Channels;
        public Resampler(float[] taps, int interp, int decim, int channels = 1)
        {
            if (taps == null) throw new ArgumentNullException(nameof(taps));
            if (taps.Length == 0) throw new ArgumentException("Prototype taps must not be empty.", nameof(taps));
            if (taps.Length > 16384) throw new ArgumentOutOfRangeException(nameof(taps), "At most 16384 prototype taps.");
            if (interp < 1 || interp > 1024) throw new ArgumentOutOfRangeException(nameof(interp), "interp must be from 1 to 1024.");
            if (decim < 1 || decim > 1024) throw new ArgumentOutOfRangeException(nameof(decim), "decim must be from 1 to 1024.");
            if ((taps.Length + interp - 1) / interp > 64)
                throw new ArgumentOutOfRangeException(nameof(taps), "At most 64 taps per branch (taps.Length <= 64 * interp).");
            if (channels < 1 || channels > 16384) throw new ArgumentOutOfRangeException(nameof(channels), "From 1 to 16384 channels.");
            foreach (var t in taps)
                if (!float.IsFinite(t)) throw new ArgumentOutOfRangeException(nameof(taps), "Taps must be finite.");
            IntPtr h;
            fixed (float* t = taps)
                QpskCuda.Check(QpskCuda.qpsk_resamp_create(t, taps.Length, interp, decim, channels, out h), nameof(taps));
            _o = new QpskHandle(h, QpskCuda.qpsk_resamp_destroy);
            Interp = interp;
            Decim = decim;
            Channels = channels;
        }
        // iqIn: [Channels][nFloats] interleaved IQ, nFloats = iqIn.Length / Channels; iqOut: [Channels][outStrideFloats].
        // Returns floats written per channel.
        public long Process(ReadOnlySpan<float> iqIn, Span<float> iqOut, long outStrideFloats)
        {
            if (iqIn.Length % (2 * Channels) != 0)
                throw new ArgumentException("Input must be Channels rows of interleaved IQ with even length.", nameof(iqIn));
            if (outStrideFloats < 0 || iqOut.Length < Channels * outStrideFloats)
                throw new ArgumentException("Output span is too small for Channels rows of outStrideFloats.", nameof(iqOut));
            long n;
            fixed (float* i = iqIn) fixed (float* o = iqOut)
                QpskCuda.Check(QpskCuda.qpsk_resamp_process(_h, i, iqIn.Length / Channels, o, outStrideFloats, out n), nameof(iqOut));
            GC.KeepAlive(this);
            return n;
        }
        public void Reset()
        {
            QpskCuda.Check(QpskCuda.qpsk_resamp_reset(_h));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    // Rate-1/2 K = 7 convolutional encoder (generators 171, 133 octal; not in the reference, definition in qpskcuda.h):
    // Channels streams of bits as 0/1 bytes, each input bit -> the pair (c0, c1), one QPSK symbol.  The register persists
    // across calls: any chunking gives the same bits.
    public sealed unsafe class ConvEncoder : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int Channels;
        public ConvEncoder(int channels = 1)
        {
            if (channels < 1 || channels > 16384) throw new ArgumentOutOfRangeException(nameof(channels), "From 1 to 16384 channels.");
            IntPtr h;
            QpskCuda.Check(QpskCuda.qpsk_conv_create(channels, out h), nameof(channels));
            _o = new QpskHandle(h, QpskCuda.qpsk_conv_destroy);
            Channels = channels;
        }
        // bits: [Channels][nBits] 0/1 bytes, nBits = bits.Length / Channels; coded: [Channels][2 * nBits]
        public void Encode(ReadOnlySpan<byte> bits, Span<byte> coded)
        {
            if (bits.Length % Channels != 0) throw new ArgumentException("Input must be Channels rows of equal length.", nameof(bits));
            if (coded.Length < 2 * bits.Length) throw new ArgumentException("Output must hold two bits per input bit.", nameof(coded));
            fixed (byte* i = bits) fixed (byte* o = coded)
                QpskCuda.Check(QpskCuda.qpsk_conv_encode(_h, i, bits.Length / Channels, o), nameof(bits));
            GC.KeepAlive(this);
        }
        public void Reset()
        {
            QpskCuda.Check(QpskCuda.qpsk_conv_reset(_h));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    // Batched soft-decision Viterbi decoder of ConvEncoder's code (not in the reference; exact rules in qpskcuda.h): Costas
    // output symbols in (deModulateConstellation), decided bits as 0/1 bytes out, one trellis step per symbol.  Bits come out
    // in blocks of 32, 64 steps behind the newest symbol; Flush emits the rest and resets the decoder.
    public sealed unsafe class ViterbiDecoder : IDisposable
    {
        public const float ScaleCoherent = 32.0f;       // QPSK_VITERBI_SCALE_COHERENT
        public const float ScaleDifferential = 24.0f;   // QPSK_VITERBI_SCALE_DIFFERENTIAL
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int Channels;
        public ViterbiDecoder(int channels = 1, bool differential = true, float scale = 0.0f)
        {
            if (channels < 1 || channels > 16384) throw new ArgumentOutOfRangeException(nameof(channels), "From 1 to 16384 channels.");
            if (scale == 0.0f) scale = differential ? ScaleDifferential : ScaleCoherent;
            if (!(scale > 0.0f) || !float.IsFinite(scale)) throw new ArgumentOutOfRangeException(nameof(scale), "scale must be finite and > 0.");
            IntPtr h;
            QpskCuda.Check(QpskCuda.qpsk_viterbi_create(channels, differential ? 1 : 0, scale, out h), nameof(scale));
            _o = new QpskHandle(h, QpskCuda.qpsk_viterbi_destroy);
            Channels = channels;
        }
        public long BitsBound(long maxSymbols)
        {
            QpskCuda.Check(QpskCuda.qpsk_viterbi_bits_bound(_h, maxSymbols, out long cap), nameof(maxSymbols));
            GC.KeepAlive(this);
            return cap;
        }
        // symIQ: [Channels][symStrideFloats] interleaved IQ, nSym[c] symbols used per row; bits: [Channels][bitsCap] with
        // bitsCap >= BitsBound(max nSym); nBits[c] receives the bits written per row.
        public void Decode(ReadOnlySpan<float> symIQ, long symStrideFloats, ReadOnlySpan<long> nSym, Span<byte> bits, long bitsCap, Span<long> nBits)
            => Run(false, symIQ, symStrideFloats, nSym, bits, bitsCap, nBits);
        public void Flush(ReadOnlySpan<float> symIQ, long symStrideFloats, ReadOnlySpan<long> nSym, Span<byte> bits, long bitsCap, Span<long> nBits)
            => Run(true, symIQ, symStrideFloats, nSym, bits, bitsCap, nBits);
        void Run(bool flush, ReadOnlySpan<float> symIQ, long symStrideFloats, ReadOnlySpan<long> nSym, Span<byte> bits, long bitsCap, Span<long> nBits)
        {
            if (symStrideFloats < 0 || (symStrideFloats & 1) != 0 || symIQ.Length < Channels * symStrideFloats)
                throw new ArgumentException("Symbols must be Channels rows of symStrideFloats (even) floats.", nameof(symIQ));
            if (nSym.Length < Channels || nBits.Length < Channels) throw new ArgumentException("One count per channel.", nameof(nSym));
            if (bitsCap < 0 || bits.Length < Channels * bitsCap) throw new ArgumentException("Output span is too small for Channels rows of bitsCap.", nameof(bits));
            fixed (float* s = symIQ) fixed (long* ns = nSym) fixed (byte* b = bits) fixed (long* nb = nBits)
                QpskCuda.Check(flush ? QpskCuda.qpsk_viterbi_flush(_h, s, symStrideFloats, ns, b, bitsCap, nb)
                                     : QpskCuda.qpsk_viterbi_decode(_h, s, symStrideFloats, ns, b, bitsCap, nb), nameof(bits));
            GC.KeepAlive(this);
        }
        public void Reset()
        {
            QpskCuda.Check(QpskCuda.qpsk_viterbi_reset(_h));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    // One frame found by FrameSync (qpsk_fsync_frame): the window was multiplied by j^-Rotation.
    [StructLayout(LayoutKind.Sequential)]
    public struct SyncedFrame
    {
        public long Position;   // p*, the absolute symbol index of the frame's first coded symbol
        public int Metric, Energy, Rotation, Channel;
    }

    // Soft-decision frame synchronizer for coded frames (not in the reference; exact rules in qpskcuda.h): correlates the
    // encoded start of a frame (32 zero bits and START) against the Costas output and cuts one window of WindowSymbols per
    // frame, derotated by the lock phase it found in coherent mode.  Windows go to a ViterbiDecoder of Channels * slots
    // rows (Flush), the payload starts at PayloadBitOffset of its bits, and ReedSolomon decodes it.
    public sealed unsafe class FrameSync : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int Channels, PatternSymbols, FrameSymbols, WindowSymbols, Rho;
        public int PayloadBitOffset => PatternSymbols;
        public FrameSync(int channels, bool differential, ReadOnlySpan<byte> startMarker, int payloadBytes, int nEnd, float scale = 0.0f, int rho = 0)
        {
            if (channels < 1 || channels > 16384) throw new ArgumentOutOfRangeException(nameof(channels), "From 1 to 16384 channels.");
            if (startMarker.Length < 1 || startMarker.Length > 24) throw new ArgumentOutOfRangeException(nameof(startMarker), "START must be 1 to 24 bytes.");
            if (scale == 0.0f) scale = differential ? ViterbiDecoder.ScaleDifferential : ViterbiDecoder.ScaleCoherent;
            IntPtr h;
            fixed (byte* s = startMarker)
                QpskCuda.Check(QpskCuda.qpsk_fsync_create(channels, differential ? 1 : 0, scale, s, startMarker.Length, payloadBytes, nEnd, rho, out h), nameof(payloadBytes));
            _o = new QpskHandle(h, QpskCuda.qpsk_fsync_destroy);
            Channels = channels;
            QpskCuda.Check(QpskCuda.qpsk_fsync_shape(h, out PatternSymbols, out FrameSymbols, out WindowSymbols, out Rho));
        }
        public long SlotsBound(long maxSymbols)
        {
            QpskCuda.Check(QpskCuda.qpsk_fsync_slots_bound(_h, maxSymbols, out long slots), nameof(maxSymbols));
            GC.KeepAlive(this);
            return slots;
        }
        // symIQ: [Channels][symStrideFloats] interleaved IQ, nSym[c] symbols per row; slot c * slots + j receives the j-th
        // frame channel c completes: frames [Channels * slots][frameStrideFloats], frameNSym / nBytes / info per slot (0 and
        // Position -1 in an empty slot).  slots >= SlotsBound(max nSym), frameStrideFloats >= 2 * WindowSymbols.
        public void Process(ReadOnlySpan<float> symIQ, long symStrideFloats, ReadOnlySpan<long> nSym, int slots, Span<float> frames,
                            long frameStrideFloats, Span<int> frameNSym, Span<long> nBytes, Span<SyncedFrame> info)
        {
            if (symStrideFloats < 0 || (symStrideFloats & 1) != 0 || symIQ.Length < Channels * symStrideFloats)
                throw new ArgumentException("Symbols must be Channels rows of symStrideFloats (even) floats.", nameof(symIQ));
            if (nSym.Length < Channels) throw new ArgumentException("One count per channel.", nameof(nSym));
            long n = (long)Channels * slots;
            if (slots < 0 || frames.Length < n * frameStrideFloats || frameNSym.Length < n || nBytes.Length < n || info.Length < n)
                throw new ArgumentException("Output spans are too small for Channels * slots slots.", nameof(frames));
            fixed (float* s = symIQ) fixed (long* ns = nSym) fixed (float* f = frames) fixed (int* fn = frameNSym)
            fixed (long* nb = nBytes) fixed (SyncedFrame* inf = info)
                QpskCuda.Check(QpskCuda.qpsk_fsync_process(_h, s, symStrideFloats, ns, slots, f, frameStrideFloats, fn, nb, (IntPtr)inf, out long _), nameof(slots));
            GC.KeepAlive(this);
        }
        public void Reset()
        {
            QpskCuda.Check(QpskCuda.qpsk_fsync_reset(_h));
            GC.KeepAlive(this);
        }
        public void Dispose() => _o.Dispose();
    }

    // Reed-Solomon outer code over GF(2^8) with depth-interleaved blocks (not in the reference; exact definition and
    // decoding rule in qpskcuda.h): Nroots parity bytes per K message bytes, N = K + Nroots <= 255, T = Nroots / 2 byte
    // errors corrected per codeword, Depth codewords interleaved byte by byte per block of BlockBytes.  Stateless: calls
    // may run on any stream in any order.
    public sealed unsafe class ReedSolomon : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public readonly int Nroots, K, Depth;
        public int N => K + Nroots;
        public int T => Nroots / 2;
        public int BlockBytes => Depth * N;
        public ReedSolomon(int nroots = 32, int k = 223, int depth = 1)
        {
            if (nroots < 2 || nroots > 32 || (nroots & 1) != 0) throw new ArgumentOutOfRangeException(nameof(nroots), "nroots must be even, from 2 to 32.");
            if (k < 1 || k + nroots > 255) throw new ArgumentOutOfRangeException(nameof(k), "k must be >= 1 with k + nroots <= 255.");
            if (depth < 1 || depth > 8) throw new ArgumentOutOfRangeException(nameof(depth), "From 1 to 8 codewords per block.");
            IntPtr h;
            QpskCuda.Check(QpskCuda.qpsk_rs_create(nroots, k, depth, out h), nameof(nroots));
            _o = new QpskHandle(h, QpskCuda.qpsk_rs_destroy);
            Nroots = nroots; K = k; Depth = depth;
        }
        // message: whole blocks of Depth * K bytes -> code: Depth * N bytes per block
        public byte[] Encode(ReadOnlySpan<byte> message)
        {
            if (message.Length % (Depth * K) != 0) throw new ArgumentException("Message must be whole blocks of Depth * K bytes.", nameof(message));
            long nBlocks = message.Length / (Depth * K);
            var code = new byte[nBlocks * BlockBytes];
            fixed (byte* m = message) fixed (byte* c = code)
                QpskCuda.Check(QpskCuda.qpsk_rs_encode(_h, m, nBlocks, c), nameof(message));
            GC.KeepAlive(this);
            return code;
        }
        // code: whole blocks (a remainder is ignored) -> message bytes; status: one per codeword in block order, the bytes
        // corrected or -1 where the codeword passed through uncorrected
        public byte[] Decode(ReadOnlySpan<byte> code, out int[] status)
        {
            long nBlocks = code.Length / BlockBytes;
            var message = new byte[nBlocks * Depth * K];
            status = new int[nBlocks * Depth];
            fixed (byte* c = code) fixed (byte* m = message) fixed (int* s = status)
                QpskCuda.Check(QpskCuda.qpsk_rs_decode(_h, c, nBlocks, m, s), nameof(code));
            GC.KeepAlive(this);
            return message;
        }
        public void Dispose() => _o.Dispose();
    }
}

namespace QPSK
{
    public sealed unsafe class QPSKModulator : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public long baudRate;                                                        // QPSKModulator.cs:34
        public QPSKModulator(int SampleRate, int SymbolRate, double RrcAlpha = 0.9, int rrcSpan = 6,
                             bool differentialEncoding = true, string? tsc = null)   // :18
        {
            baudRate = 2L * SymbolRate / 8L;
            QpskCuda.Check(QpskCuda.qpsk_mod_create(SampleRate, SymbolRate, RrcAlpha, rrcSpan, differentialEncoding ? 1 : 0, tsc, out IntPtr h));
            _o = new QpskHandle(h, QpskCuda.qpsk_mod_destroy);
        }
        public double[] getCoeef()                                                   // :32
        {
            QpskCuda.Check(QpskCuda.qpsk_mod_taps(_h, null, 0, out int n));
            var h = new double[n];
            fixed (double* p = h) QpskCuda.Check(QpskCuda.qpsk_mod_taps(_h, p, n, out n));
            GC.KeepAlive(this);
            return h;
        }
        public float[] ModulateBytes(ReadOnlySpan<byte> payload, ReadOnlySpan<byte> startMarker, ReadOnlySpan<byte> endMarker,
                                     bool pulseShaping = true)                      // :54  framing START|payload|END on the device
        {
            if (startMarker.Length == 0) throw new ArgumentException("startMarker cannot be empty.", nameof(startMarker));   // :60
            if (endMarker.Length == 0) throw new ArgumentException("endMarker cannot be empty.", nameof(endMarker));         // :61
            int ps = pulseShaping ? 1 : 0;
            fixed (byte* p = payload) fixed (byte* s = startMarker) fixed (byte* e = endMarker)
            {
                QpskCuda.Check(QpskCuda.qpsk_mod_modulate_bytes(_h, p, payload.Length, s, startMarker.Length, e, endMarker.Length, ps,
                                                                null, 0, out long n));
                var y = new float[n];
                if (n > 0)
                    fixed (float* o = y)
                        QpskCuda.Check(QpskCuda.qpsk_mod_modulate_bytes(_h, p, payload.Length, s, startMarker.Length, e, endMarker.Length,
                                                                        ps, o, n, out n));
                GC.KeepAlive(this);
                return y;
            }
        }
        public float[] ModulateTextUtf8(string text, string startMarker = "\u0002", string endMarker = "\u0003",
                                        bool pulseShaping = true, Encoding? encoding = null)   // :74  stays managed + ModulateBytes
        {
            if (text == null) throw new ArgumentNullException(nameof(text));         // :81
            encoding ??= Encoding.UTF8;
            // GetBytes(null) throws ArgumentNullException, as upstream (:85-86)
            return ModulateBytes(encoding.GetBytes(text), encoding.GetBytes(startMarker), encoding.GetBytes(endMarker), pulseShaping);
        }
        public float[] Modulate(string data, bool pulseShaping = true)              // :104
        {
            if (data == null) throw new ArgumentNullException(nameof(data));
            byte[] bits = Encoding.Latin1.GetBytes(data);                            // one char per bit, as upstream
            int ps = pulseShaping ? 1 : 0;
            fixed (byte* b = bits)
            {
                QpskCuda.Check(QpskCuda.qpsk_mod_modulate_bits(_h, b, bits.Length, ps, null, 0, out long n));
                var y = new float[n];
                if (n > 0)
                    fixed (float* o = y)
                        QpskCuda.Check(QpskCuda.qpsk_mod_modulate_bits(_h, b, bits.Length, ps, o, n, out n));
                GC.KeepAlive(this);
                return y;
            }
        }
        public void Dispose() => _o.Dispose();
    }

    public sealed unsafe class QPSKDeModulator : IDisposable
    {
        readonly QpskHandle _o;
        IntPtr _h => _o.Ptr;
        public QPSKDeModulator(int SampleRate, int SymbolRate, float RrcAlpha = 0.9f, int rrcSpan = 6,
                               double SymbolSyncBandwith = 0.0001, double CostasLoopBandwith = 120, double CFOLoopBandwith = 0.0001f,
                               bool differentialEncoding = true, string? tsc = null)   // QPSKDeModulator.cs:11
        {
            // use_fll = 0: the fll.Process call is commented out upstream (:359, :435); max_frame_bytes = 0: library default
            QpskCuda.Check(QpskCuda.qpsk_demod_create(SampleRate, SymbolRate, RrcAlpha, rrcSpan, SymbolSyncBandwith, CostasLoopBandwith,
                                                      CFOLoopBandwith, differentialEncoding ? 1 : 0, tsc, 0, 0, out IntPtr h));
            _o = new QpskHandle(h, QpskCuda.qpsk_demod_destroy);
        }
        // opt-in CMA equalizer between clock recovery and Costas (not in the reference; nTaps 0 = off, the default)
        public void SetEqualizer(int nTaps, float mu, float modulus = 1.0f)
        {
            QpskCuda.Check(QpskCuda.qpsk_demod_set_equalizer(_h, nTaps, mu, modulus));
            _eqTaps = nTaps;
            GC.KeepAlive(this);
        }
        int _eqTaps;
        public float[] EqualizerTaps()
        {
            var t = new float[2 * _eqTaps];
            fixed (float* p = t) QpskCuda.Check(QpskCuda.qpsk_demod_equalizer_taps(_h, p, t.Length));
            GC.KeepAlive(this);
            return t;
        }
        // opt-in feed-forward AGC ahead of the FLL and the matched filter (not in the reference; window 0 = off, the default)
        public void SetAgc(int window, float refLevel = 1.0f, float maxGain = 65536.0f)
        {
            QpskCuda.Check(QpskCuda.qpsk_demod_set_agc(_h, window, refLevel, maxGain));
            GC.KeepAlive(this);
        }
        // opt-in fractionally spaced CMA equalizer between the matched filter and clock recovery (not in the reference;
        // needs SampleRate / SymbolRate an integer 2..8; nTaps 0 = off, the default)
        public void SetFractionalEqualizer(int nTaps, float mu, float modulus = 1.0f)
        {
            QpskCuda.Check(QpskCuda.qpsk_demod_set_fractional_equalizer(_h, nTaps, mu, modulus));
            _fseTaps = nTaps;
            GC.KeepAlive(this);
        }
        int _fseTaps;
        public float[] FractionalEqualizerTaps()
        {
            var t = new float[2 * _fseTaps];
            fixed (float* p = t) QpskCuda.Check(QpskCuda.qpsk_demod_fractional_equalizer_taps(_h, p, t.Length));
            GC.KeepAlive(this);
            return t;
        }
        public byte[] DeModulateBytes(ReadOnlySpan<float> samplesIQ, ReadOnlySpan<byte> startMarker, ReadOnlySpan<byte> endMarker)   // :169
        {
            if (startMarker.Length == 0) throw new ArgumentException("startMarker cannot be empty.", nameof(startMarker));   // :174
            if (endMarker.Length == 0) throw new ArgumentException("endMarker cannot be empty.", nameof(endMarker));         // :175
            if ((samplesIQ.Length & 1) != 0)
                throw new ArgumentException("Samples must be interleaved IQ with even length.", nameof(samplesIQ));         // :347-348 via :177
            var buf = new byte[samplesIQ.Length / 8 + 64];                            // what this call's samples alone can carry
            fixed (float* i = samplesIQ) fixed (byte* s = startMarker) fixed (byte* e = endMarker) fixed (byte* o = buf)
            {
                int st = QpskCuda.qpsk_demod_bytes(_h, i, samplesIQ.Length, s, startMarker.Length, e, endMarker.Length, o, buf.Length,
                                                   out long n);
                if (st == -6)
                {
                    // QPSK_ERR_CAPACITY: the frame accumulated on the device over earlier calls (MTU-block streaming) and is
                    // longer than this call's buffer; it is still in the framer ring, fetch it at its reported size
                    var big = new byte[n];
                    fixed (byte* b = big) QpskCuda.Check(QpskCuda.qpsk_demod_last_payload(_h, b, big.Length, out n));
                    GC.KeepAlive(this);
                    return big;
                }
                QpskCuda.Check(st, nameof(samplesIQ));
                GC.KeepAlive(this);
                if (n == 0) return Array.Empty<byte>();                              // :180, :258
                var payload = new byte[n];
                Array.Copy(buf, payload, n);
                return payload;
            }
        }
        public string DeModulateTextUtf8(ReadOnlySpan<float> samplesIQ, string startMarker = "\u0002", string endMarker = "\u0003",
                                         Encoding? encoding = null)                 // :262
        {
            encoding ??= Encoding.UTF8;
            byte[] p = DeModulateBytes(samplesIQ, encoding.GetBytes(startMarker), encoding.GetBytes(endMarker));
            return p.Length == 0 ? string.Empty : encoding.GetString(p);
        }
        public string DeModulate(float[] SamplesIQ)                                  // :339
        {
            if (SamplesIQ == null) throw new ArgumentNullException(nameof(SamplesIQ));   // :341
            return DeModulate(SamplesIQ.AsSpan());
        }
        public string DeModulate(ReadOnlySpan<float> SamplesIQ)                      // :345  '0'/'1' chars, TSC already stripped
        {
            if ((SamplesIQ.Length & 1) != 0)
                throw new ArgumentException("Samples must be interleaved IQ with even length.", nameof(SamplesIQ));   // :347-348
            if (SamplesIQ.Length == 0) return "";                                    // :350-351
            var buf = new byte[Math.Max(SamplesIQ.Length, 16)];
            fixed (float* i = SamplesIQ) fixed (byte* o = buf)
            {
                QpskCuda.Check(QpskCuda.qpsk_demod_bits(_h, i, SamplesIQ.Length, o, buf.Length, out long n), nameof(SamplesIQ));
                GC.KeepAlive(this);
                return Encoding.ASCII.GetString(buf, 0, (int)n);
            }
        }
        public float[] deModulateConstellation(ReadOnlySpan<float> SamplesIQ)        // :427
        {
            if ((SamplesIQ.Length & 1) != 0)
                throw new ArgumentException("Samples must be interleaved IQ with even length.", nameof(SamplesIQ));   // :430
            var buf = new float[Math.Max(SamplesIQ.Length, 2)];
            fixed (float* i = SamplesIQ) fixed (float* o = buf)
            {
                QpskCuda.Check(QpskCuda.qpsk_demod_constellation(_h, i, SamplesIQ.Length, o, buf.Length, out long nSym), nameof(SamplesIQ));
                GC.KeepAlive(this);
                var y = new float[nSym << 1];                                        // :446
                Array.Copy(buf, y, y.Length);
                return y;
            }
        }
        public void Dispose() => _o.Dispose();
    }
}
