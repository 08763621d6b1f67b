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
        n = x.shape[-1] if x.ndim == 2 else x.size
        if iqOut is None:
            iqOut = np.empty(x.shape if out_len is None else out_len, np.float32)
        cap = iqOut.shape[-1] if iqOut.ndim == 2 else iqOut.size
        check(lib().qpsk_fir_filter(self._h, _ptr(x), _ptr(iqOut), n, cap))
        return iqOut

    def fftFilter(self, iqData) -> np.ndarray:
        """fftFilter(float[]) :96-141."""
        if iqData is None:
            raise ArgumentNullException("iqData")
        x = _f32(iqData)
        n = x.shape[-1] if x.ndim == 2 else x.size
        y = np.empty(x.shape if n % 2 == 0 else 0, np.float32)
        check(lib().qpsk_fir_fft_filter(self._h, _ptr(x), _ptr(y), n))
        return y

    def Decimate(self, iqIn, decim: int, out_cap_floats=None):
        """Decimate-by-D matched filter (north_star (2)): Filter() kept at stream indices 0, D, 2D, ... across calls.
        Returns the kept samples (interleaved IQ; [channels, n] for batch handles)."""
        x = _f32(iqIn)
        n = x.shape[-1] if x.ndim == 2 else x.size
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
        n = x.shape[-1] if x.ndim == 2 else x.size
        y = outputIQ if outputIQ is not None else np.empty(x.shape if out_len is None else out_len, np.float32)
        cap = y.shape[-1] if y.ndim == 2 else y.size
        check(lib().qpsk_fll_process(self._h, _ptr(x), _ptr(y), n, cap))
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
        n = x.shape[-1] if x.ndim == 2 else x.size
        ns = np.zeros(self.channels, np.int32)
        if outputSymbolsIQ is not None:
            y = outputSymbolsIQ
            cap = y.shape[-1] if y.ndim == 2 else y.size
            check(lib().qpsk_mm_process(self._h, _ptr(x), n, _ptr(y), cap, ns.ctypes.data_as(N.i32p)))
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
        n = x.shape[-1] if x.ndim == 2 else x.size
        y = iqOut if iqOut is not None else np.empty(x.shape if out_len is None else out_len, np.float32)
        cap = y.shape[-1] if y.ndim == 2 else y.size
        check(lib().qpsk_costas_process(self._h, _ptr(x), _ptr(y), n, cap))
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
        n = x.shape[-1] if x.ndim == 2 else x.size
        y = iqOut if iqOut is not None else np.empty(x.shape, np.float32)
        cap = y.shape[-1] if y.ndim == 2 else y.size
        check(lib().qpsk_eq_process(self._h, _ptr(x), _ptr(y), n, cap))
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
