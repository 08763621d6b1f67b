"""Host-side mirror of the reference's class surface over the C ABI (include/qpskcuda.h).

Same class and method names, argument meaning and error behaviour as the C# classes
(RRCFilter, ComplexFIRFilter, FLLBandEdgeFilter, MuellerMuller, CostasLoopQpsk, QPSKModulator,
QPSKDeModulator), so the parity tests read like the reference's own usage.  numpy arrays stand in
for Span<float>; `*_dev` methods take raw device pointers (e.g. torch.Tensor.data_ptr()).
Everything computes on the GPU through libqpskcuda.so; nothing here falls back to the CPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from ._native import (ArgumentException, ArgumentNullException, ArgumentOutOfRangeException, ChanParams,  # noqa: F401
                      QpskCudaError, check, lib)

FIR_FAST, FIR_EXACT, FIR_FMA, FIR_SPLIT = N.FIR_FAST, N.FIR_EXACT, N.FIR_FMA, N.FIR_SPLIT


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a: np.ndarray):
    return C.c_void_p(a.ctypes.data)


def _bytes_arr(b) -> np.ndarray:
    return np.frombuffer(bytes(b), dtype=np.uint8).copy() if len(b) else np.zeros(0, np.uint8)


def _iq(x) -> np.ndarray:
    """complex64 samples or interleaved float32 IQ -> contiguous interleaved float32 IQ"""
    a = np.asarray(x)
    return np.ascontiguousarray(a, np.complex64).view(np.float32) if np.iscomplexobj(a) else _f32(a)


def _row_floats(a: np.ndarray) -> int:
    """floats per channel of a [channels, n] batch, or of a 1-D array"""
    return a.shape[-1] if a.ndim == 2 else a.size


def _sym_counts(n_sym, channels: int, stride: int) -> np.ndarray:
    """int64 symbols used per channel: all `stride` floats of each row, or `n_sym` broadcast to every channel"""
    if n_sym is None:
        return np.full(channels, stride // 2, np.int64)
    return np.ascontiguousarray(np.broadcast_to(np.asarray(n_sym, np.int64), (channels,)))


def _bank_process(fn, h, a: np.ndarray, n_floats: int, rows: int, out_stride: int) -> np.ndarray:
    """The host call of the blocks whose output count depends on their state: without `out_stride` the call is asked for
    the floats per output row first (its QPSK_ERR_CAPACITY answer) -> complex64 [rows, n_out]."""
    n = C.c_int64(0)
    if not out_stride:
        st = fn(h, None, n_floats, None, -1, C.byref(n))
        if st != N.ERR_CAPACITY:
            check(st)
        out_stride = n.value
    y = np.zeros((rows, max(out_stride, 0)), np.float32)
    check(fn(h, _ptr(a), n_floats, _ptr(y), out_stride, C.byref(n)))
    return np.ascontiguousarray(y[:, : n.value]).view(np.complex64)


# ---- library / device ---------------------------------------------------------------------
def device_count() -> int:
    n = C.c_int(0)
    check(lib().qpsk_device_count(C.byref(n)))
    return n.value


def set_device(ordinal: int):
    check(lib().qpsk_set_device(ordinal))


def device_info() -> dict:
    sm, ma, mi, mem = C.c_int(), C.c_int(), C.c_int(), C.c_int64()
    check(lib().qpsk_device_info(C.byref(sm), C.byref(ma), C.byref(mi), C.byref(mem)))
    return dict(sm_count=sm.value, cc=(ma.value, mi.value), hbm_bytes=mem.value)


def launch_count() -> int:
    return int(lib().qpsk_launch_count())


def launch_count_reset():
    lib().qpsk_launch_count_reset()


def measure_fma_peak() -> float:
    t = C.c_double(0)
    check(lib().qpsk_measure_fma_peak(C.byref(t)))
    return t.value


class PinnedBuffer:
    """qpsk_host_alloc'd float32 buffer exposed as a numpy array (what a C# caller would wrap in a Span)."""

    def __init__(self, n_floats: int):
        self._p = C.c_void_p()
        check(lib().qpsk_host_alloc(C.byref(self._p), n_floats * 4))
        self.array = np.ctypeslib.as_array(C.cast(self._p, N.f32p), shape=(n_floats,))

    def free(self):
        if self._p:
            lib().qpsk_host_free(self._p)
            self._p = None
            self.array = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class RegisteredArray:
    """Page-lock a caller-owned contiguous numpy array in place (qpsk_host_register) — the Python stand-in for a C#
    float[] held by a pinned GCHandle.  Use as a context manager or call release()."""

    def __init__(self, array: np.ndarray):
        if not array.flags["C_CONTIGUOUS"]:
            raise N.ArgumentException("array must be contiguous")
        self.array = array
        self._p = array.ctypes.data
        check(lib().qpsk_host_register(self._p, array.nbytes))

    def release(self):
        if self._p:
            lib().qpsk_host_unregister(self._p)
            self._p = None

    def __enter__(self):
        return self.array

    def __exit__(self, *exc):
        self.release()

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


def fill_uniform_dev(seed: int, stream_id: int, first: int, n: int, d_out: int, stream: int = 0):
    check(lib().qpsk_fill_uniform_dev(seed, stream_id, first, n, d_out, stream))


# ---- a1 -------------------------------------------------------------------------------------
class RRCFilter:
    @staticmethod
    def generateCoefficents(spanSymbols: float, beta: float, sampleRate: int, SymbolRate: int) -> np.ndarray:
        n = C.c_int(0)
        check(lib().qpsk_rrc_taps(spanSymbols, beta, sampleRate, SymbolRate, None, 0, C.byref(n)))
        out = np.empty(max(n.value, 0), np.float64)
        check(lib().qpsk_rrc_taps(spanSymbols, beta, sampleRate, SymbolRate, out.ctypes.data_as(N.f64p), n.value, C.byref(n)))
        return out


def real_taps_to_iq(h) -> np.ndarray:
    """ToInterleavedIQRealTaps (MS/QPSKDeModulator.cs:278-288)."""
    t = np.zeros(2 * len(h), np.float32)
    t[0::2] = np.asarray(h, np.float64).astype(np.float32)
    return t


class _Handle:
    _destroy = None

    def __init__(self):
        self._h = C.c_void_p()

    def close(self):
        if self._h and self._destroy:
            getattr(lib(), self._destroy)(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---- a2-a5 ----------------------------------------------------------------------------------
class ComplexFIRFilter(_Handle):
    """ComplexFIRFilter (MS/Models/FIRFilter.cs:8-232) on the GPU."""
    _destroy = "qpsk_fir_destroy"

    def __init__(self, tapsInterleavedIQ, channels: int = 1):
        super().__init__()
        if tapsInterleavedIQ is None:
            raise ArgumentNullException("tapsInterleavedIQ")
        t = _f32(tapsInterleavedIQ)
        self.taps = t.copy()
        self.channels = channels
        check(lib().qpsk_fir_create_batch(t.ctypes.data_as(N.f32p), t.size, channels, C.byref(self._h)))

    def set_mode(self, mode: int):
        check(lib().qpsk_fir_set_mode(self._h, mode))

    def reset(self):
        check(lib().qpsk_fir_reset(self._h))

    def last_kernel(self) -> str:
        buf = C.create_string_buffer(128)
        check(lib().qpsk_fir_last_kernel(self._h, buf, 128))
        return buf.value.decode()

    def Filter(self, iqIn, iqOut=None, out_len=None) -> np.ndarray:
        """Filter(ReadOnlySpan<float>, Span<float>) :80-91.  Batch handles: shape [channels, n_floats]."""
        x = _f32(iqIn)
        n = _row_floats(x)
        if iqOut is None:
            iqOut = np.empty(x.shape if out_len is None else out_len, np.float32)
        check(lib().qpsk_fir_filter(self._h, _ptr(x), _ptr(iqOut), n, _row_floats(iqOut)))
        return iqOut

    def fftFilter(self, iqData) -> np.ndarray:
        """fftFilter(float[]) :96-141."""
        if iqData is None:
            raise ArgumentNullException("iqData")
        x = _f32(iqData)
        n = _row_floats(x)
        y = np.empty(x.shape if n % 2 == 0 else 0, np.float32)
        check(lib().qpsk_fir_fft_filter(self._h, _ptr(x), _ptr(y), n))
        return y

    def Decimate(self, iqIn, decim: int, out_cap_floats=None):
        """Decimate-by-D matched filter (north_star (2)): Filter() kept at stream indices 0, D, 2D, ... across calls.
        Returns the kept samples (interleaved IQ; [channels, n] for batch handles)."""
        x = _f32(iqIn)
        n = _row_floats(x)
        cap = (2 * ((n // 2 + decim - 1) // max(decim, 1)) + 2) if out_cap_floats is None else out_cap_floats
        y = np.zeros((self.channels, max(cap, 0)), np.float32)
        no = C.c_int64(0)
        check(lib().qpsk_fir_decimate(self._h, _ptr(x), n, decim, _ptr(y), cap, C.byref(no)))
        y = y[:, : no.value]
        return y[0].copy() if self.channels == 1 and x.ndim == 1 else y.copy()

    def decimate_dev(self, d_in: int, n_floats: int, decim: int, d_out: int, out_cap_floats: int, in_stride: int = 0,
                     out_stride: int = 0, stream: int = 0) -> int:
        no = C.c_int64(0)
        check(lib().qpsk_fir_decimate_dev(self._h, d_in, n_floats, in_stride or n_floats, decim, d_out, out_cap_floats,
                                          out_stride or out_cap_floats, C.byref(no), stream))
        return no.value

    def filter_dev(self, d_in: int, d_out: int, n_floats: int, in_stride: int = 0, out_stride: int = 0, stream: int = 0):
        check(lib().qpsk_fir_filter_dev(self._h, d_in, d_out, n_floats, in_stride or n_floats, out_stride or n_floats, stream))

    def fft_filter_dev(self, d_in: int, d_out: int, n_floats: int, in_stride: int = 0, out_stride: int = 0, stream: int = 0):
        check(lib().qpsk_fir_fft_filter_dev(self._h, d_in, d_out, n_floats, in_stride or n_floats, out_stride or n_floats, stream))

    def get_state(self) -> np.ndarray:
        keep = self.taps.size // 2 - 1
        out = np.empty((self.channels, 2 * keep), np.float32)
        check(lib().qpsk_fir_get_state(self._h, out.ctypes.data_as(N.f32p), out.size))
        return out

    def set_state(self, hist):
        h = _f32(hist)
        check(lib().qpsk_fir_set_state(self._h, h.ctypes.data_as(N.f32p), h.size))


# ---- a7-a8 ----------------------------------------------------------------------------------
def fll_design(sps: float, rolloff: float, filterSize: int):
    """DesignFilter (MS/Models/Band-Edge Filter.cs:132-183): (lower_iq, upper_iq)."""
    lo = np.empty(2 * max(filterSize, 0), np.float32)
    up = np.empty(2 * max(filterSize, 0), np.float32)
    check(lib().qpsk_fll_design(sps, rolloff, filterSize, lo.ctypes.data_as(N.f32p), up.ctypes.data_as(N.f32p)))
    return lo, up


class FLLBandEdgeFilter(_Handle):
    """FLLBandEdgeFilter (MS/Models/Band-Edge Filter.cs:14-203) on the GPU: 8 lanes per stream (the reference's 8 SIMD lanes), a chain warp and a side warp per four streams (csrc/fll_duo.cu)."""
    _destroy = "qpsk_fll_destroy"

    def __init__(self, sps, rolloff, filterSize, bandwidth, channels: int = 1):
        super().__init__()
        self.sps, self.rolloff, self.filterSize, self.bandwidth = sps, rolloff, filterSize, bandwidth   # public fields :19-22
        self.channels = channels
        self._design = (sps, rolloff, filterSize)
        check(lib().qpsk_fll_create_batch(sps, rolloff, filterSize, bandwidth, channels, C.byref(self._h)))

    def taps(self):
        return fll_design(*self._design)

    def Process(self, inputIQ, outputIQ=None, out_len=None):
        """Process(float[]) :90-96 -> the output array; with `outputIQ` given it is Process(ReadOnlySpan<float>,
        Span<float>) :64-87: writes into the caller's array and returns the number of COMPLEX samples processed (:71, :86)."""
        x = _f32(inputIQ)
        n = _row_floats(x)
        y = outputIQ if outputIQ is not None else np.empty(x.shape if out_len is None else out_len, np.float32)
        check(lib().qpsk_fll_process(self._h, _ptr(x), _ptr(y), n, _row_floats(y)))
        return (n >> 1) if outputIQ is not None else y

    def process_dev(self, d_in, d_out, n_floats, in_stride=0, out_stride=0, stream=0):
        check(lib().qpsk_fll_process_dev(self._h, d_in, d_out, n_floats, in_stride or n_floats, out_stride or n_floats, stream))

    @property
    def state(self):
        p = np.empty(self.channels, np.float32)
        f = np.empty(self.channels, np.float32)
        check(lib().qpsk_fll_get_state(self._h, p.ctypes.data_as(N.f32p), f.ctypes.data_as(N.f32p)))
        return (float(p[0]), float(f[0])) if self.channels == 1 else (p, f)

    @state.setter
    def state(self, pf):
        p = _f32(np.broadcast_to(np.asarray(pf[0], np.float32), (self.channels,)))
        f = _f32(np.broadcast_to(np.asarray(pf[1], np.float32), (self.channels,)))
        check(lib().qpsk_fll_set_state(self._h, p.ctypes.data_as(N.f32p), f.ctypes.data_as(N.f32p)))

    # the reference's public loop-state fields (Band-Edge Filter.cs:25-26), readable and writable between calls
    @property
    def phase(self):
        return self.state[0]

    @phase.setter
    def phase(self, v):
        self.state = (v, self.state[1])

    @property
    def freq(self):
        return self.state[1]

    @freq.setter
    def freq(self, v):
        self.state = (self.state[0], v)


# ---- a9 ---------------------------------------------------------------------------------------
class MuellerMuller(_Handle):
    """MuellerMuller (MS/Models/MuellerMuller.cs:17-250) on the GPU."""
    _destroy = "qpsk_mm_destroy"

    def __init__(self, samplesPerSymbol, kp, ki, channels: int = 1):
        super().__init__()
        self.channels = channels
        check(lib().qpsk_mm_create_batch(samplesPerSymbol, kp, ki, channels, C.byref(self._h)))

    def Process(self, incomingMfSamplesIQ, outputSymbolsIQ=None, cap_floats=None):
        """Process(float[]) :141-157 -> the symbols (interleaved IQ, `n << 1` floats; batch handles: list of per-channel
        arrays).  With `outputSymbolsIQ` given it is Process(ReadOnlySpan<float>, Span<float>) :52-136: writes into the
        caller's array ([channels][cap] for batch handles) and returns outSymbols, the number of complex SYMBOLS written
        (:135; an int for one channel, an int array per channel for batch handles)."""
        x = _f32(incomingMfSamplesIQ)
        n = _row_floats(x)
        ns = np.zeros(self.channels, np.int32)
        if outputSymbolsIQ is not None:
            y = outputSymbolsIQ
            check(lib().qpsk_mm_process(self._h, _ptr(x), n, _ptr(y), _row_floats(y), ns.ctypes.data_as(N.i32p)))
            return int(ns[0]) if self.channels == 1 else ns
        cap = n if cap_floats is None else cap_floats
        y = np.zeros((self.channels, max(cap, 0)), np.float32)
        check(lib().qpsk_mm_process(self._h, _ptr(x), n, _ptr(y), cap, ns.ctypes.data_as(N.i32p)))
        outs = [y[c, : int(ns[c]) << 1].copy() for c in range(self.channels)]
        return outs[0] if self.channels == 1 else outs

    @property
    def state(self):
        b = np.empty(self.channels, np.int32)
        q = np.empty(self.channels, np.int32)
        mu = np.empty(self.channels, np.float64)
        it = np.empty(self.channels, np.float64)
        check(lib().qpsk_mm_get_state(self._h, b.ctypes.data_as(N.i32p), mu.ctypes.data_as(N.f64p),
                                      it.ctypes.data_as(N.f64p), q.ctypes.data_as(N.i32p)))
        if self.channels == 1:
            return dict(baseIndex=int(b[0]), mu=float(mu[0]), ncoIntegral=float(it[0]), queued=int(q[0]))
        return dict(baseIndex=b, mu=mu, ncoIntegral=it, queued=q)


def mm_gains_from_bw(sym_bw: float):
    kp, ki = C.c_double(), C.c_double()
    check(lib().qpsk_mm_gains_from_bw(sym_bw, C.byref(kp), C.byref(ki)))
    return kp.value, ki.value


# ---- a10 --------------------------------------------------------------------------------------
class CostasLoopQpsk(_Handle):
    """CostasLoopQpsk (MS/Models/CostasLoopQpsk.cs:19-131) on the GPU."""
    _destroy = "qpsk_costas_destroy"

    def __init__(self, sampleRate, loopBandwidthHz, damping=0.707, channels: int = 1):
        super().__init__()
        self.channels = channels
        check(lib().qpsk_costas_create_batch(sampleRate, loopBandwidthHz, damping, channels, C.byref(self._h)))

    def Process(self, iqIn, iqOut=None, out_len=None):
        """Process(float[]) :119-125 -> the output array; with `iqOut` given it is Process(ReadOnlySpan<float>, Span<float>)
        :98-114: writes into the caller's array and returns the number of COMPLEX samples processed (:105, :113)."""
        x = _f32(iqIn)
        n = _row_floats(x)
        y = iqOut if iqOut is not None else np.empty(x.shape if out_len is None else out_len, np.float32)
        check(lib().qpsk_costas_process(self._h, _ptr(x), _ptr(y), n, _row_floats(y)))
        return (n >> 1) if iqOut is not None else y

    @staticmethod
    def GetSign(i, q):
        """GetSign :52-56 — (di, dq) = (+-1, +-1), zero counts as positive."""
        return (1.0 if np.float32(i) >= 0 else -1.0), (1.0 if np.float32(q) >= 0 else -1.0)

    def GetState(self):
        t = np.empty(self.channels, np.float64)
        f = np.empty(self.channels, np.float64)
        check(lib().qpsk_costas_get_state(self._h, t.ctypes.data_as(N.f64p), f.ctypes.data_as(N.f64p)))
        return (float(t[0]), float(f[0])) if self.channels == 1 else (t, f)


# ---- blind CMA equalizer (not in the reference) ------------------------------------------------
class CmaEqualizer(_Handle):
    """Blind CMA equalizer on the GPU (csrc/eq.cu; arithmetic spec in include/qpskcuda.h): `n_taps` complex taps (1..64)
    adapted by the constant-modulus rule with step `mu` towards |y|^2 = `modulus`, one output per input, group delay
    (n_taps-1)//2 inputs.  `sps` 1 (the default) is symbol-spaced; `sps` 2..8 makes it fractionally spaced on a T/sps-spaced
    input, the taps updating on every sps-th sample of the stream.  State persists across calls."""
    _destroy = "qpsk_eq_destroy"

    def __init__(self, n_taps: int, mu: float, modulus: float = 1.0, channels: int = 1, sps: int = 1):
        super().__init__()
        self.n_taps, self.channels, self.sps = n_taps, channels, sps
        check(lib().qpsk_eq_create_fractional(n_taps, mu, modulus, sps, channels, C.byref(self._h)))

    def Process(self, iqIn, iqOut=None):
        """-> the equalized symbols (interleaved IQ; [channels, n_floats] for batch handles).  With `iqOut` given the
        outputs go there and the number of complex symbols processed is returned."""
        x = _f32(iqIn)
        n = _row_floats(x)
        y = iqOut if iqOut is not None else np.empty(x.shape, np.float32)
        check(lib().qpsk_eq_process(self._h, _ptr(x), _ptr(y), n, _row_floats(y)))
        return (n >> 1) if iqOut is not None else y

    def process_dev(self, d_in: int, d_out: int, n_floats: int, in_stride: int = 0, out_stride: int = 0, d_n_sym: int = 0,
                    stream: int = 0):
        check(lib().qpsk_eq_process_dev(self._h, d_in, d_out, n_floats, in_stride or n_floats, out_stride or n_floats,
                                        d_n_sym or None, stream))

    @property
    def taps(self) -> np.ndarray:
        """[2*n_taps] interleaved IQ ([channels, 2*n_taps] for batch handles)."""
        out = np.empty((self.channels, 2 * self.n_taps), np.float32)
        check(lib().qpsk_eq_get_taps(self._h, out.ctypes.data_as(N.f32p), out.size))
        return out[0] if self.channels == 1 else out

    @taps.setter
    def taps(self, t):
        t = _f32(t)
        check(lib().qpsk_eq_set_taps(self._h, t.ctypes.data_as(N.f32p), t.size))

    def reset(self):
        check(lib().qpsk_eq_reset(self._h))


# ---- feed-forward AGC (not in the reference) -----------------------------------------------------
class Agc(_Handle):
    """Feed-forward AGC on the GPU (csrc/agc.cu; definition in include/qpskcuda.h): per channel, each sample is scaled by
    fminf(ref / m, max_gain), m the peak of max(|re|, |im|) over a `window`-sample window (1..4096) that looks window-1
    samples ahead of it, so the output is the input delayed by window-1 samples, at level `ref`.  State persists across
    calls: any chunking of the stream gives the same outputs bit for bit."""
    _destroy = "qpsk_agc_destroy"

    def __init__(self, window: int, ref: float = 1.0, max_gain: float = 65536.0, channels: int = 1):
        super().__init__()
        self.window, self.channels = window, channels
        check(lib().qpsk_agc_create_batch(window, ref, max_gain, channels, C.byref(self._h)))

    def process(self, x) -> np.ndarray:
        """x: complex64 [channels, n] (or [n] for one channel; interleaved float32 IQ also taken) -> complex64 outputs of
        the same shape, one per input sample."""
        a = _iq(x)
        rows = a.reshape(self.channels, -1)
        y = np.empty(rows.shape, np.float32)
        check(lib().qpsk_agc_process(self._h, _ptr(rows), _ptr(y), rows.shape[1], rows.shape[1]))
        out = y.view(np.complex64)
        return out[0] if (self.channels == 1 and a.ndim == 1) else out

    def process_dev(self, d_in: int, d_out: int, n_floats: int, in_stride: int = 0, out_stride: int = 0, stream: int = 0):
        """Device pointers: [channels][in_stride] floats -> [channels][out_stride], n_floats per channel (strides in
        floats, 0 = n_floats).  d_out must not overlap d_in."""
        check(lib().qpsk_agc_process_dev(self._h, d_in, d_out, n_floats, in_stride or n_floats, out_stride or n_floats,
                                         stream))

    @property
    def gain(self) -> np.ndarray:
        """float32 [channels]: the gain of each channel's last output (max_gain before any sample)."""
        out = np.empty(self.channels, np.float32)
        check(lib().qpsk_agc_gain(self._h, out.ctypes.data_as(N.f32p), out.size))
        return out

    def gain_dev(self, d_gain: int, stream: int = 0):
        """Copy the last gains to d_gain[channels] (float32, device) in stream order."""
        check(lib().qpsk_agc_gain_dev(self._h, d_gain, stream))

    def reset(self):
        check(lib().qpsk_agc_reset(self._h))


# ---- polyphase analysis channelizer (not in the reference) -------------------------------------
def pfb_taps(channels: int, taps_per_branch: int, cutoff: float, atten_db: float = 60.0) -> np.ndarray:
    """Kaiser-windowed sinc prototype for PfbChannelizer (fp64, unit DC gain, channels*taps_per_branch taps); cutoff in
    cycles per input sample, e.g. 0.5/channels for adjacent channels meeting at their -6 dB points."""
    n = C.c_int(0)
    check(lib().qpsk_pfb_taps(channels, taps_per_branch, cutoff, atten_db, None, 0, C.byref(n)))
    out = np.empty(n.value, np.float64)
    check(lib().qpsk_pfb_taps(channels, taps_per_branch, cutoff, atten_db, out.ctypes.data_as(N.f64p), n.value, C.byref(n)))
    return out


class PfbChannelizer(_Handle):
    """Critically sampled polyphase analysis channelizer on the GPU (csrc/pfb.cu; definition in include/qpskcuda.h): one
    wideband stream in, `channels` (a power of two, 2..1024) channel streams out at 1/channels of the rate, channel k
    centred at +k/channels cycles per input sample.  `taps`: the real prototype (e.g. pfb_taps(...)), at most
    32*channels taps.  State persists across calls: any chunking of the stream gives the same outputs."""
    _destroy = "qpsk_pfb_destroy"

    def __init__(self, taps, channels: int):
        super().__init__()
        if taps is None:
            raise ArgumentNullException("taps")
        t = _f32(taps)
        self.channels = channels
        check(lib().qpsk_pfb_create(t.ctypes.data_as(N.f32p), t.size, channels, C.byref(self._h)))

    def process(self, x, out_stride: int = 0) -> np.ndarray:
        """x: complex64 samples (or interleaved float32 IQ) of the wideband stream -> complex64 [channels, n_out], the
        outputs this call completes.  `out_stride` (floats) sizes the output rows like the C call; 0 = just enough."""
        a = _iq(x)
        return _bank_process(lib().qpsk_pfb_process, self._h, a, a.size, self.channels, out_stride)

    def process_dev(self, d_in: int, n_floats: int, d_out: int, out_stride: int, stream: int = 0) -> int:
        """Device pointers: n_floats of the wideband stream -> d_out [channels][out_stride] floats.  Returns the floats
        written per channel (the n_floats to pass to QPSKDeModulator.demod_bytes_dev with in_stride = out_stride)."""
        n = C.c_int64(0)
        check(lib().qpsk_pfb_process_dev(self._h, d_in, n_floats, d_out, out_stride, C.byref(n), stream))
        return n.value

    def reset(self):
        check(lib().qpsk_pfb_reset(self._h))


# ---- digital down-converter bank (not in the reference) ----------------------------------------
class DdcBank(_Handle):
    """Frequency-translating decimating filter bank on the GPU (csrc/ddc.cu; definition in include/qpskcuda.h): one
    wideband stream in, one channel per entry of `freqs` (cycles per input sample, each in [-0.5, 0.5), 1..2048 of them)
    out at 1/`decim` of the rate, channel k mixed down by freqs[k], filtered with the real prototype `taps` (1..4096 taps,
    e.g. scipy.signal.firwin) and decimated.  State persists across calls: any chunking of the stream gives the same
    outputs."""
    _destroy = "qpsk_ddc_destroy"

    def __init__(self, taps, freqs, decim: int):
        super().__init__()
        if taps is None:
            raise ArgumentNullException("taps")
        if freqs is None:
            raise ArgumentNullException("freqs")
        t = _f32(taps)
        f = np.ascontiguousarray(freqs, dtype=np.float64).ravel()
        self.channels = f.size
        self.decim = decim
        check(lib().qpsk_ddc_create(t.ctypes.data_as(N.f32p), t.size, f.ctypes.data_as(N.f64p), f.size, decim,
                                    C.byref(self._h)))

    def process(self, x, out_stride: int = 0) -> np.ndarray:
        """x: complex64 samples (or interleaved float32 IQ) of the wideband stream -> complex64 [channels, n_out], the
        outputs this call completes.  `out_stride` (floats) sizes the output rows like the C call; 0 = just enough."""
        a = _iq(x)
        return _bank_process(lib().qpsk_ddc_process, self._h, a, a.size, self.channels, out_stride)

    def process_dev(self, d_in: int, n_floats: int, d_out: int, out_stride: int, stream: int = 0) -> int:
        """Device pointers: n_floats of the wideband stream -> d_out [channels][out_stride] floats.  Returns the floats
        written per channel (the n_floats to pass to QPSKDeModulator.demod_bytes_dev with in_stride = out_stride)."""
        n = C.c_int64(0)
        check(lib().qpsk_ddc_process_dev(self._h, d_in, n_floats, d_out, out_stride, C.byref(n), stream))
        return n.value

    def reset(self):
        check(lib().qpsk_ddc_reset(self._h))


# ---- rational resampler (not in the reference) --------------------------------------------------
class Resampler(_Handle):
    """Batched rational resampler on the GPU (csrc/resamp.cu; definition in include/qpskcuda.h): `channels` streams, each
    interpolated by `interp` (L), filtered with the real prototype `taps` and decimated by `decim` (M), i.e.
    scipy.signal.upfirdn(taps, x, L, M) per channel, streamed.  No L factor: taps summing to L (e.g.
    L * scipy.signal.firwin(..., scale=True)) pass a carrier with unit gain.  L, M in 1..1024, 1..16384 taps with
    ceil(len(taps) / L) <= 64.  State persists across calls: any chunking of the stream gives the same outputs."""
    _destroy = "qpsk_resamp_destroy"

    def __init__(self, taps, interp: int, decim: int, channels: int = 1):
        super().__init__()
        if taps is None:
            raise ArgumentNullException("taps")
        t = _f32(taps).ravel()
        self.interp, self.decim, self.channels = interp, decim, channels
        check(lib().qpsk_resamp_create(t.ctypes.data_as(N.f32p), t.size, interp, decim, channels, C.byref(self._h)))

    def process(self, x, out_stride: int = 0) -> np.ndarray:
        """x: complex64 [channels, n] (or [n] for one channel; interleaved float32 IQ also taken) -> complex64
        [channels, n_out] (or [n_out]), the outputs this call completes.  `out_stride` (floats) sizes the output rows like
        the C call; 0 = just enough."""
        a = _iq(x)
        rows = a.reshape(self.channels, -1)
        out = _bank_process(lib().qpsk_resamp_process, self._h, rows, rows.shape[1], self.channels, out_stride)
        return out[0] if (self.channels == 1 and a.ndim == 1) else out

    def process_dev(self, d_in: int, n_floats: int, d_out: int, out_stride: int, in_stride: int = 0,
                    stream: int = 0) -> int:
        """Device pointers: [channels][in_stride] floats (0 = n_floats), n_floats per channel -> d_out
        [channels][out_stride].  Returns the floats written per channel (the n_floats to pass to
        QPSKDeModulator.demod_bytes_dev with in_stride = out_stride)."""
        n = C.c_int64(0)
        check(lib().qpsk_resamp_process_dev(self._h, d_in, n_floats, in_stride or n_floats, d_out, out_stride,
                                            C.byref(n), stream))
        return n.value

    def reset(self):
        check(lib().qpsk_resamp_reset(self._h))


# ---- convolutional code and Viterbi decoder (not in the reference) --------------------------------
VITERBI_SCALE_COHERENT = 32.0          # QPSK_VITERBI_SCALE_COHERENT: symbols at unit amplitude (DESIGN.md §3 K13)
VITERBI_SCALE_DIFFERENTIAL = 24.0      # QPSK_VITERBI_SCALE_DIFFERENTIAL


class ConvEncoder(_Handle):
    """Rate-1/2 K = 7 convolutional encoder (generators 171, 133 octal; csrc/fec.cu, definition in include/qpskcuda.h),
    `channels` streams of bits as 0/1 bytes.  Each input bit gives the pair (c0, c1), c0 first; one pair is one QPSK
    symbol.  The register persists across calls: any chunking gives the same bits."""
    _destroy = "qpsk_conv_destroy"

    def __init__(self, channels: int = 1):
        super().__init__()
        self.channels = channels
        check(lib().qpsk_conv_create(channels, C.byref(self._h)))

    def encode(self, bits) -> np.ndarray:
        """bits: uint8 0/1 [channels, n] (or [n] for one channel) -> uint8 [channels, 2n] (or [2n])."""
        a = np.ascontiguousarray(bits, np.uint8)
        rows = a.reshape(self.channels, -1)
        out = np.zeros((self.channels, 2 * rows.shape[1]), np.uint8)
        check(lib().qpsk_conv_encode(self._h, _ptr(rows), rows.shape[1], _ptr(out)))
        return out[0] if (self.channels == 1 and a.ndim == 1) else out

    def encode_dev(self, d_bits: int, n_bits: int, d_out: int, out_stride: int, bits_stride: int = 0, stream: int = 0):
        """Device pointers: [channels][bits_stride] (0 = n_bits) -> d_out [channels][out_stride], 2 * n_bits per row."""
        check(lib().qpsk_conv_encode_dev(self._h, d_bits, n_bits, bits_stride or n_bits, d_out, out_stride, stream))

    def reset(self):
        check(lib().qpsk_conv_reset(self._h))


class ViterbiDecoder(_Handle):
    """Batched soft-decision Viterbi decoder of ConvEncoder's code (csrc/fec.cu; exact rules in include/qpskcuda.h): the
    Costas output of every channel (QPSKDeModulator.constellation_dev) in, decided bits as 0/1 bytes out, one trellis step
    per symbol.  `differential` decodes the differential map without a phase reference; `scale` (None = the default of
    the mode) maps unit-amplitude symbols to int8 soft values.  Bits come out in blocks of 32, 64 steps behind the newest
    symbol; flush() emits the rest and resets the handle."""
    _destroy = "qpsk_viterbi_destroy"

    def __init__(self, channels: int = 1, differential: bool = True, scale: float = None):
        super().__init__()
        if scale is None:
            scale = VITERBI_SCALE_DIFFERENTIAL if differential else VITERBI_SCALE_COHERENT
        self.channels, self.differential, self.scale = channels, bool(differential), float(scale)
        check(lib().qpsk_viterbi_create(channels, int(differential), scale, C.byref(self._h)))

    def bits_bound(self, max_sym: int) -> int:
        b = C.c_int64(0)
        check(lib().qpsk_viterbi_bits_bound(self._h, max_sym, C.byref(b)))
        return b.value

    def _host(self, fn, sym, n_sym):
        if sym is None:
            sym = np.zeros((self.channels, 0), np.complex64)
        rows = np.ascontiguousarray(_iq(sym).reshape(self.channels, -1))
        stride = rows.shape[1]
        ns = _sym_counts(n_sym, self.channels, stride)
        cap = self.bits_bound(int(ns.max()) if ns.size else 0)
        out = np.zeros((self.channels, cap), np.uint8)
        nb = np.zeros(self.channels, np.int64)
        check(getattr(lib(), fn)(self._h, _ptr(rows), stride, _ptr(ns), _ptr(out), cap, _ptr(nb)))
        outs = [out[c, : nb[c]].copy() for c in range(self.channels)]
        return outs[0] if (self.channels == 1 and np.ndim(sym) == 1) else outs

    def decode(self, sym, n_sym=None):
        """sym: complex64 [channels, n] (or [n]; interleaved float32 IQ also taken), n_sym: symbols used per channel
        (default all) -> per channel the uint8 0/1 bits this call completes (a list, or one array for a 1-D input)."""
        return self._host("qpsk_viterbi_decode", sym, n_sym)

    def flush(self, sym=None, n_sym=None):
        """decode(), then every bit not yet emitted; the handle is reset afterwards."""
        return self._host("qpsk_viterbi_flush", sym, n_sym)

    def decode_dev(self, d_sym: int, sym_stride: int, d_n_sym: int, d_bits: int, bits_cap: int, d_n_bits: int,
                   stream: int = 0):
        """Device pointers: d_sym [channels][sym_stride] floats with int32 d_n_sym[channels] (what
        QPSKDeModulator.constellation_dev writes) -> d_bits [channels][bits_cap] uint8, int64 d_n_bits[channels].
        bits_cap >= bits_bound(sym_stride // 2)."""
        check(lib().qpsk_viterbi_decode_dev(self._h, d_sym, sym_stride, d_n_sym, d_bits, bits_cap, d_n_bits, stream))

    def flush_dev(self, d_sym: int, sym_stride: int, d_n_sym: int, d_bits: int, bits_cap: int, d_n_bits: int,
                  stream: int = 0):
        check(lib().qpsk_viterbi_flush_dev(self._h, d_sym, sym_stride, d_n_sym, d_bits, bits_cap, d_n_bits, stream))

    def reset(self):
        check(lib().qpsk_viterbi_reset(self._h))


# ---- Reed-Solomon outer code (not in the reference) ------------------------------------------------
class ReedSolomon(_Handle):
    """Reed-Solomon code over GF(2^8) with depth-I byte interleaving (csrc/rs.cu; exact definition and decoding rule in
    include/qpskcuda.h): `nroots` parity bytes (t = nroots / 2 correctable byte errors) per `k` message bytes, n = k +
    nroots <= 255, `depth` codewords interleaved byte by byte per block.  The outer code around ConvEncoder /
    ViterbiDecoder: transmit coded_frame_bits(rs.encode(payload), START, END); receive constellation_dev ->
    ViterbiDecoder.flush_dev -> frame_bits_dev -> decode_dev.  The handle holds constants only: calls may run on any
    stream in any order."""
    _destroy = "qpsk_rs_destroy"

    def __init__(self, nroots: int = 32, k: int = 223, depth: int = 1):
        super().__init__()
        self.nroots, self.k, self.depth = nroots, k, depth
        check(lib().qpsk_rs_create(nroots, k, depth, C.byref(self._h)))

    @property
    def n(self) -> int:
        return self.k + self.nroots

    @property
    def t(self) -> int:
        return self.nroots // 2

    @property
    def block_bytes(self) -> int:
        """code bytes per block, depth * n (depth * k of them the message)"""
        return self.depth * self.n

    def encode(self, msg) -> bytes:
        """whole blocks of message bytes (a multiple of depth * k) -> their code bytes"""
        a = _bytes_arr(msg)
        mb = self.depth * self.k
        if a.size % mb:
            raise ArgumentException(f"message length {a.size} is not a multiple of depth * k = {mb}")
        out = np.zeros(a.size // mb * self.block_bytes, np.uint8)
        check(lib().qpsk_rs_encode(self._h, _ptr(a), a.size // mb, _ptr(out)))
        return out.tobytes()

    def decode(self, code):
        """code bytes (whole blocks; a remainder is ignored) -> (message bytes, int32 status per codeword in block order:
        the number of bytes corrected, or -1 where the codeword was not within t and passes through as received)"""
        a = _bytes_arr(code)
        nb = a.size // self.block_bytes
        out = np.zeros(nb * self.depth * self.k, np.uint8)
        st = np.zeros(nb * self.depth, np.int32)
        check(lib().qpsk_rs_decode(self._h, _ptr(a), nb, _ptr(out), _ptr(st)))
        return out.tobytes(), st

    def encode_dev(self, d_msg: int, msg_stride: int, rows: int, n_blocks: int, d_code: int, code_stride: int,
                   stream: int = 0):
        """Device pointers: n_blocks blocks in every row, d_msg [rows][msg_stride] -> d_code [rows][code_stride]."""
        check(lib().qpsk_rs_encode_dev(self._h, d_msg, msg_stride, rows, n_blocks, d_code, code_stride, stream))

    def decode_dev(self, d_code: int, code_stride: int, d_n_bytes: int, rows: int, d_msg: int, msg_stride: int,
                   d_n_msg: int, d_status: int, status_stride: int, stream: int = 0):
        """Device pointers, the payload rows QPSKDeModulator.frame_bits_dev / demod_bytes_dev write: d_code
        [rows][code_stride] with int64 d_n_bytes[rows] -> d_msg [rows][msg_stride], int64 d_n_msg[rows], int32 d_status
        [rows][status_stride]; every row decodes its whole blocks.  msg_stride >= (code_stride // block_bytes) * depth * k,
        status_stride >= (code_stride // block_bytes) * depth."""
        check(lib().qpsk_rs_decode_dev(self._h, d_code, code_stride, d_n_bytes, rows, d_msg, msg_stride, d_n_msg, d_status,
                                       status_stride, stream))


# ---- soft-decision frame synchronizer for coded frames (not in the reference) ------------------------------------------
FSYNC_RHO_DEFAULT = 144                # QPSK_FSYNC_RHO_DEFAULT (DESIGN.md §3 K15)
FSYNC_INFO = np.dtype([("position", "<i8"), ("metric", "<i4"), ("energy", "<i4"), ("rotation", "<i4"),
                       ("channel", "<i4")])                     # qpsk_fsync_frame


class FrameSync(_Handle):
    """Soft-decision frame synchronizer for the coded frames of modem.coded_frame_bits (csrc/fsync.cu; exact rules in
    include/qpskcuda.h): it correlates the known encoded start (32 zero bits and `start_marker`, P symbols) against the
    soft values of the Costas output, and cuts one window of F + delta symbols per frame (delta = 1 differential, 0
    coherent), derotated by the Costas lock phase it found in coherent mode.  `payload_bytes` and `n_end` (the END
    marker's length) fix F; `rho` (0 = the default) is the detection threshold in 1/256 of the energy.  Receive path:
    constellation_dev -> process_dev -> ViterbiDecoder(channels * slots).flush_dev -> pack_bits from payload_bit_offset
    -> ReedSolomon.decode_dev.  State is carried per channel: any chunking of a stream gives the same frames."""
    _destroy = "qpsk_fsync_destroy"

    def __init__(self, channels: int = 1, differential: bool = True, start_marker: bytes = b"START",
                 payload_bytes: int = 64, n_end: int = 3, scale: float = None, rho: int = 0):
        super().__init__()
        if scale is None:
            scale = VITERBI_SCALE_DIFFERENTIAL if differential else VITERBI_SCALE_COHERENT
        s = _bytes_arr(start_marker)
        self.channels, self.differential, self.scale = channels, bool(differential), float(scale)
        self.start_marker, self.payload_bytes, self.n_end = bytes(start_marker), payload_bytes, n_end
        check(lib().qpsk_fsync_create(channels, int(differential), scale, _ptr(s), s.size, payload_bytes, n_end, rho,
                                      C.byref(self._h)))
        v = [C.c_int(0) for _ in range(4)]
        check(lib().qpsk_fsync_shape(self._h, *(C.byref(x) for x in v)))
        self.pattern_syms, self.frame_syms, self.window_syms, self.rho = (x.value for x in v)

    @property
    def payload_bit_offset(self) -> int:
        """where the payload starts in the F bits ViterbiDecoder.flush_dev emits for a window: past the 32 lead bits and
        START, which are the P pattern symbols"""
        return self.pattern_syms

    def layout(self) -> dict:
        """P (pattern symbols), F (frame symbols), the window length F + delta, the payload bit offset and rho"""
        return dict(P=self.pattern_syms, F=self.frame_syms, window=self.window_syms,
                    payload_bit_offset=self.payload_bit_offset, rho=self.rho)

    def slots_bound(self, max_sym: int) -> int:
        b = C.c_int64(0)
        check(lib().qpsk_fsync_slots_bound(self._h, max_sym, C.byref(b)))
        return b.value

    def process(self, sym, n_sym=None):
        """sym: complex64 [channels, n] (or [n]; interleaved float32 IQ also taken), n_sym: symbols used per channel
        (default all) -> per channel the frames this call completes, a list of (window complex64 [F + delta], info
        record of FSYNC_INFO); a list per channel, or one list for a 1-D input."""
        rows = np.ascontiguousarray(_iq(sym).reshape(self.channels, -1))
        stride = rows.shape[1]
        ns = _sym_counts(n_sym, self.channels, stride)
        slots = self.slots_bound(int(ns.max()) if ns.size else 0)
        S, L = self.channels * slots, self.window_syms
        frames = np.zeros((max(S, 1), L), np.complex64)
        fn = np.zeros(max(S, 1), np.int32)
        nb = np.zeros(max(S, 1), np.int64)
        info = np.zeros(max(S, 1), FSYNC_INFO)
        need = C.c_int64(0)
        check(lib().qpsk_fsync_process(self._h, _ptr(rows), stride, _ptr(ns), slots, _ptr(frames), 2 * L, _ptr(fn),
                                       _ptr(nb), _ptr(info), C.byref(need)))
        outs = [[(frames[c * slots + j].copy(), info[c * slots + j]) for j in range(slots) if fn[c * slots + j] > 0]
                for c in range(self.channels)]
        return outs[0] if (self.channels == 1 and np.ndim(sym) == 1) else outs

    def process_dev(self, d_sym: int, sym_stride: int, d_n_sym: int, slots: int, d_frames: int, frame_stride: int,
                    d_frame_n_sym: int, d_n_bytes: int, d_info: int, stream: int = 0):
        """Device pointers: d_sym [channels][sym_stride] floats with int32 d_n_sym[channels] (what
        QPSKDeModulator.constellation_dev writes) -> slot c * slots + j: the j-th frame of channel c in this call, in
        d_frames [channels * slots][frame_stride] floats, int32 d_frame_n_sym, int64 d_n_bytes and d_info (FSYNC_INFO)
        per slot.  slots >= slots_bound(sym_stride // 2), frame_stride >= 2 * window_syms."""
        check(lib().qpsk_fsync_process_dev(self._h, d_sym, sym_stride, d_n_sym, slots, d_frames, frame_stride,
                                           d_frame_n_sym, d_n_bytes, d_info, stream))

    def reset(self):
        check(lib().qpsk_fsync_reset(self._h))
