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
