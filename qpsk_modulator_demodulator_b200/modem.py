"""Host-side mirror of QPSKModulator / QPSKDeModulator and the synthetic channel over the C ABI.

Same names, argument meaning and error behaviour as the C# classes (MS/QPSKModulator.cs,
MS/QPSKDeModulator.cs); the batch (`channels=`) and `*_dev` forms are the device-resident variants
the benchmarks time.  Everything computes on the GPU through libqpskcuda.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as N
from ._native import ArgumentNullException, ChanParams, check, lib
from .api import _Handle, _bytes_arr, _f32, _ptr


# ---- a6 ---------------------------------------------------------------------------------------
class FormatException(ValueError):
    """System.FormatException (BitPacker.BitsToBytes on a character other than '0' / '1')."""


class BitPacker:
    """HelperFunctions.BitPacker (MS/Models/HelperFunctions.cs:11-70): host-side string helpers, MSB first.  They stay
    host code in the C# deployment too (the device works on packed bits: qpsk_unpack_bits_dev / qpsk_pack_bits_dev and
    the framer kernel); mirrored here so that callers of the reference's helpers find them."""

    @staticmethod
    def BytesToBitString(data) -> str:                                          # :14-29
        a = np.frombuffer(bytes(data), np.uint8)
        if a.size == 0:
            return ""
        return (np.unpackbits(a) + ord("0")).astype(np.uint8).tobytes().decode("ascii")

    @staticmethod
    def BitsToBytes(bits: str, bitOffset: int) -> bytes:                        # :32-57
        if bits is None:
            raise N.ArgumentNullException("bits")
        if not 0 <= bitOffset <= 7:
            raise N.ArgumentOutOfRangeException("bitOffset")
        usable = len(bits) - bitOffset
        if usable < 8:
            return b""
        raw = np.frombuffer(bits[bitOffset: bitOffset + 8 * (usable // 8)].encode("latin-1", "replace"), np.uint8)
        if ((raw != ord("0")) & (raw != ord("1"))).any():
            raise FormatException("Bit string must contain only '0'/'1'.")
        return np.packbits(raw & 1).tobytes()

    @staticmethod
    def IndexOf(haystack, needle) -> int:                                       # :59-69
        return bytes(haystack).find(bytes(needle))


class QPSKModulator(_Handle):
    """QPSKModulator (MS/QPSKModulator.cs:18-168) on the GPU: polyphase RRC pulse shaping."""
    _destroy = "qpsk_mod_destroy"

    def __init__(self, SampleRate, SymbolRate, RrcAlpha=0.9, rrcSpan=6, differentialEncoding=True, tsc=None):
        super().__init__()
        t = None if tsc is None else tsc.encode("ascii")
        check(lib().qpsk_mod_create(SampleRate, SymbolRate, RrcAlpha, rrcSpan, int(differentialEncoding), t, C.byref(self._h)))
        self.baudRate = 2 * SymbolRate // 8                                     # QPSKModulator.cs:34 (long arithmetic)

    def getCoeef(self) -> np.ndarray:
        n = C.c_int(0)
        check(lib().qpsk_mod_taps(self._h, None, 0, C.byref(n)))
        out = np.empty(n.value, np.float64)
        check(lib().qpsk_mod_taps(self._h, out.ctypes.data_as(N.f64p), n.value, C.byref(n)))
        return out

    def Modulate(self, data: str, pulseShaping: bool = True) -> np.ndarray:
        if data is None:
            raise ArgumentNullException("data")
        b = data.encode("latin-1")
        n = C.c_int64(0)
        check(lib().qpsk_mod_modulate_bits(self._h, b, len(b), int(pulseShaping), None, 0, C.byref(n)))
        out = np.empty(n.value, np.float32)
        if n.value:
            check(lib().qpsk_mod_modulate_bits(self._h, b, len(b), int(pulseShaping), _ptr(out), out.size, C.byref(n)))
        return out

    def ModulatePacked(self, packedBits: bytes, nBits: int = None, pulseShaping: bool = True) -> np.ndarray:
        """Modulate() with the bit string packed MSB-first, 8 bits per byte (SURVEY §8f-4): identical samples to
        Modulate(BitPacker.BytesToBitString(packedBits)[:nBits])."""
        if packedBits is None:
            raise ArgumentNullException("packedBits")
        p = _bytes_arr(packedBits)
        nb = 8 * p.size if nBits is None else int(nBits)
        if nb > 8 * p.size:
            raise N.ArgumentException("nBits exceeds the packed buffer")
        n = C.c_int64(0)
        check(lib().qpsk_mod_modulate_packed(self._h, _ptr(p), nb, int(pulseShaping), None, 0, C.byref(n)))
        out = np.empty(n.value, np.float32)
        if n.value:
            check(lib().qpsk_mod_modulate_packed(self._h, _ptr(p), nb, int(pulseShaping), _ptr(out), out.size, C.byref(n)))
        return out

    def ModulateBytes(self, payload: bytes, startMarker: bytes, endMarker: bytes, pulseShaping: bool = True) -> np.ndarray:
        p, s, e = _bytes_arr(payload), _bytes_arr(startMarker), _bytes_arr(endMarker)
        n = C.c_int64(0)
        args = (self._h, _ptr(p), p.size, _ptr(s), s.size, _ptr(e), e.size, int(pulseShaping))
        check(lib().qpsk_mod_modulate_bytes(*args, None, 0, C.byref(n)))
        out = np.empty(n.value, np.float32)
        if n.value:
            check(lib().qpsk_mod_modulate_bytes(*args, _ptr(out), out.size, C.byref(n)))
        return out

    def ModulateTextUtf8(self, text: str, startMarker="\x02", endMarker="\x03", pulseShaping=True) -> np.ndarray:
        if text is None:
            raise ArgumentNullException("text")
        return self.ModulateBytes(text.encode("utf-8"), startMarker.encode("utf-8"), endMarker.encode("utf-8"), pulseShaping)

    def frame_floats(self, n_payload: int, startMarker: bytes, endMarker: bytes) -> int:
        """Floats per frame for `n_payload` payload bytes (size query of the batch entry point)."""
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        n = C.c_int64(0)
        check(lib().qpsk_mod_modulate_frames_dev(self._h, None, n_payload, 1, _ptr(s), s.size, _ptr(e), e.size, None, 0,
                                                 C.byref(n), None))
        return n.value

    def ModulateFrames(self, payloads, startMarker: bytes, endMarker: bytes, out=None, out_ptr: int = 0, out_stride_floats: int = 0):
        """ModulateBytes over a batch: payloads [frames, n_payload] uint8 (host) -> samples [frames, frame_floats] (host),
        frame groups pipelined through the device (qpsk_mod_modulate_frames).  `out_ptr` / `out_stride_floats`: write into
        caller memory (e.g. a pinned buffer) instead of allocating."""
        p = np.ascontiguousarray(payloads, dtype=np.uint8)
        frames, n_payload = p.shape
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        ff = self.frame_floats(n_payload, startMarker, endMarker)
        if out_ptr:
            dst, stride = out_ptr, out_stride_floats or ff
        else:
            if out is None:
                out = np.empty((frames, ff), np.float32)
            dst, stride = out.ctypes.data, out.shape[1]
        n = C.c_int64(0)
        check(lib().qpsk_mod_modulate_frames(self._h, _ptr(p), n_payload, frames, _ptr(s), s.size, _ptr(e), e.size, dst, stride,
                                             C.byref(n)))
        return out

    def modulate_frames_dev(self, d_payloads: int, n_payload: int, frames: int, startMarker: bytes, endMarker: bytes,
                            d_out: int, out_stride_floats: int, stream: int = 0) -> int:
        """[frames][n_payload] device bytes -> [frames][out_stride_floats] device cf32; returns floats per frame."""
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        n = C.c_int64(0)
        check(lib().qpsk_mod_modulate_frames_dev(self._h, d_payloads, n_payload, frames, _ptr(s), s.size, _ptr(e), e.size,
                                                 d_out, out_stride_floats, C.byref(n), stream))
        return n.value


# ---- a11-a12 ------------------------------------------------------------------------------------
def _decode_utf8(b: bytes) -> str:
    return b.decode("utf-8", errors="replace") if b else ""


class QPSKDeModulator(_Handle):
    """QPSKDeModulator (MS/QPSKDeModulator.cs:11-456) on the GPU, `channels` independent streams."""
    _destroy = "qpsk_demod_destroy"

    def __init__(self, SampleRate, SymbolRate, RrcAlpha=0.9, rrcSpan=6, SymbolSyncBandwith=0.0001,
                 CostasLoopBandwith=120.0, CFOLoopBandwith=float(np.float32(0.0001)), differentialEncoding=True,
                 tsc=None, use_fll=False, max_frame_bytes=0, channels: int = 1):
        super().__init__()
        self.channels = channels
        t = None if tsc is None else tsc.encode("ascii")
        check(lib().qpsk_demod_create_batch(SampleRate, SymbolRate, RrcAlpha, rrcSpan, SymbolSyncBandwith, CostasLoopBandwith,
                                            CFOLoopBandwith, int(differentialEncoding), t, int(use_fll), max_frame_bytes,
                                            channels, C.byref(self._h)))

    def set_fir_mode(self, mode: int):
        check(lib().qpsk_demod_set_fir_mode(self._h, mode))

    def set_equalizer(self, n_taps: int, mu: float, modulus: float = 1.0):
        """Opt-in CMA equalizer (api.CmaEqualizer) between Mueller-Muller and Costas, for multipath channels; n_taps 0 turns
        it off.  Resets the equalizer and leaves the other loop and framer state alone.  Its group delay is absorbed: the
        bits keep their alignment, and the last (n_taps-1)//2 symbols of a call come out at the start of the next."""
        check(lib().qpsk_demod_set_equalizer(self._h, n_taps, mu, modulus))
        self._eq_taps = n_taps

    def equalizer_taps(self) -> np.ndarray:
        """[2*n_taps] interleaved IQ ([channels, 2*n_taps] for batch handles); ArgumentException when the stage is off."""
        out = np.empty((self.channels, 2 * getattr(self, "_eq_taps", 0)), np.float32)
        check(lib().qpsk_demod_equalizer_taps(self._h, out.ctypes.data_as(N.f32p), out.size))
        return out[0] if self.channels == 1 else out

    def set_fractional_equalizer(self, n_taps: int, mu: float, modulus: float = 1.0):
        """Opt-in fractionally spaced CMA equalizer (api.CmaEqualizer with sps = fs/rs) between the matched filter and
        Mueller-Muller, so clock recovery locks on an equalized eye; n_taps 0 turns it off.  Needs fs % rs == 0 and
        fs/rs in 2..8.  Independent of set_equalizer; resets this stage only.  Its group delay of (n_taps-1)//2 samples is
        absorbed: the last (n_taps-1)//2 samples of a call reach clock recovery in the next."""
        check(lib().qpsk_demod_set_fractional_equalizer(self._h, n_taps, mu, modulus))
        self._fse_taps = n_taps

    def fractional_equalizer_taps(self) -> np.ndarray:
        """[2*n_taps] interleaved IQ ([channels, 2*n_taps] for batch handles); ArgumentException when the stage is off."""
        out = np.empty((self.channels, 2 * getattr(self, "_fse_taps", 0)), np.float32)
        check(lib().qpsk_demod_fractional_equalizer_taps(self._h, out.ctypes.data_as(N.f32p), out.size))
        return out[0] if self.channels == 1 else out

    def _in(self, SamplesIQ):
        if SamplesIQ is None:
            raise ArgumentNullException("SamplesIQ")
        x = _f32(SamplesIQ)
        n = x.shape[-1] if x.ndim == 2 else x.size
        return x, n

    def DeModulate(self, SamplesIQ):
        """-> '0'/'1' string (list of strings for batch handles)."""
        x, n = self._in(SamplesIQ)
        cap = max(n, 16)
        buf = np.zeros((self.channels, cap), np.uint8)
        nb = np.zeros(self.channels, np.int64)
        check(lib().qpsk_demod_bits(self._h, _ptr(x), n, _ptr(buf), cap, _ptr(nb)))
        outs = [buf[c, : nb[c]].tobytes().decode("ascii") for c in range(self.channels)]
        return outs[0] if self.channels == 1 else outs

    def DeModulatePacked(self, SamplesIQ):
        """DeModulate() with the bits packed MSB-first (SURVEY §8f-4) -> (bytes, n_bits) (lists for batch handles);
        a trailing incomplete byte is zero-padded on the right."""
        x, n = self._in(SamplesIQ)
        cap = max(n // 8 + 8, 8)
        buf = np.zeros((self.channels, cap), np.uint8)
        nb = np.zeros(self.channels, np.int64)
        check(lib().qpsk_demod_bits_packed(self._h, _ptr(x), n, _ptr(buf), cap, _ptr(nb)))
        outs = [(buf[c, : (nb[c] + 7) // 8].tobytes(), int(nb[c])) for c in range(self.channels)]
        return outs[0] if self.channels == 1 else outs

    def DeModulateBytes(self, samplesIQ, startMarker: bytes, endMarker: bytes, cap: int = 0):
        x, n = self._in(samplesIQ)
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        cap = cap or max(n // 8 + 64, 64)
        out = np.zeros((self.channels, cap), np.uint8)
        nb = np.zeros(self.channels, np.int64)
        st = lib().qpsk_demod_bytes(self._h, _ptr(x), n, _ptr(s), s.size, _ptr(e), e.size, _ptr(out), cap, _ptr(nb))
        out = self._refetch(st, out, nb)
        outs = [out[c, : nb[c]].tobytes() for c in range(self.channels)]
        return outs[0] if self.channels == 1 else outs

    def DeModulateBytesCs16(self, samplesCs16, scale: float, startMarker: bytes, endMarker: bytes, cap: int = 0):
        """DeModulateBytes on CS16 samples (int16 I, Q pairs; [channels, n] for batch handles), widened on the device as
        (float)v * scale: half the host-to-device bytes of the cf32 call, identical payloads when the cf32 samples are
        exactly int16 * scale."""
        x = np.ascontiguousarray(samplesCs16, dtype=np.int16)
        n = x.shape[-1] if x.ndim == 2 else x.size
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        cap = cap or max(n // 8 + 64, 64)
        out = np.zeros((self.channels, cap), np.uint8)
        nb = np.zeros(self.channels, np.int64)
        st = lib().qpsk_demod_bytes_cs16(self._h, _ptr(x), n, scale, _ptr(s), s.size, _ptr(e), e.size, _ptr(out), cap, _ptr(nb))
        out = self._refetch(st, out, nb)
        outs = [out[c, : nb[c]].tobytes() for c in range(self.channels)]
        return outs[0] if self.channels == 1 else outs

    def demod_bytes_host_ptr(self, in_ptr: int, n_floats: int, startMarker: bytes, endMarker: bytes, out: np.ndarray, nb: np.ndarray,
                             cs16_scale: float = None):
        """The raw host entry point on caller-owned memory (pinned / registered / pageable): in_ptr -> [channels][n_floats]
        float32 (or int16 when cs16_scale is given), payloads into out [channels, cap], lengths into nb.  Returns the status."""
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        if cs16_scale is None:
            return lib().qpsk_demod_bytes(self._h, in_ptr, n_floats, _ptr(s), s.size, _ptr(e), e.size, _ptr(out), out.shape[1], _ptr(nb))
        return lib().qpsk_demod_bytes_cs16(self._h, in_ptr, n_floats, cs16_scale, _ptr(s), s.size, _ptr(e), e.size, _ptr(out),
                                           out.shape[1], _ptr(nb))

    def _refetch(self, st, out, nb):
        """A frame that accumulated on the device over several calls can be longer than a buffer sized from this call's
        samples (the MTU-block loop of TB/SDR/ModDemodOverSDR.cs:127-136): on QPSK_ERR_CAPACITY the completed frames are
        still in the framer ring, so they are fetched again into a buffer of the reported size instead of being lost."""
        if st != N.ERR_CAPACITY:
            check(st)
            return out
        cap = int(nb.max())
        out = np.zeros((self.channels, cap), np.uint8)
        check(lib().qpsk_demod_last_payload(self._h, _ptr(out), cap, _ptr(nb)))
        return out

    def FrameBits(self, bits, startMarker: bytes, endMarker: bytes, cap: int = 0):
        """The framer half of DeModulateBytes (MS/QPSKDeModulator.cs:182-259) on bits already demodulated: a '0'/'1'
        string (one channel) or a list of them (one per channel, lengths may differ).  Shares the framer state with
        DeModulateBytes."""
        rows = [bits] if isinstance(bits, (str, bytes)) else list(bits)
        if len(rows) != self.channels:
            raise N.ArgumentException("one bit string per channel")
        nb_in = np.array([len(r) for r in rows], np.int64)
        ld = max(int(nb_in.max()), 1)
        b = np.zeros((self.channels, ld), np.uint8)
        for c, r in enumerate(rows):
            raw = np.frombuffer(r.encode("ascii") if isinstance(r, str) else bytes(r), np.uint8)
            b[c, : raw.size] = raw & 1                       # '0' = 0x30, '1' = 0x31
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        cap = cap or max(ld // 8 + 64, 64)
        out = np.zeros((self.channels, cap), np.uint8)
        nb = np.zeros(self.channels, np.int64)
        st = lib().qpsk_demod_frame_bits(self._h, _ptr(b), ld, _ptr(nb_in), _ptr(s), s.size, _ptr(e), e.size, _ptr(out), cap, _ptr(nb))
        out = self._refetch(st, out, nb)
        outs = [out[c, : nb[c]].tobytes() for c in range(self.channels)]
        return outs[0] if self.channels == 1 else outs

    def DeModulateTextUtf8(self, samplesIQ, startMarker="\x02", endMarker="\x03"):
        p = self.DeModulateBytes(samplesIQ, startMarker.encode("utf-8"), endMarker.encode("utf-8"))
        return _decode_utf8(p) if self.channels == 1 else [_decode_utf8(b) for b in p]

    def deModulateConstellation(self, SamplesIQ):
        x, n = self._in(SamplesIQ)
        cap = max(n, 2)
        y = np.zeros((self.channels, cap), np.float32)
        ns = np.zeros(self.channels, np.int64)
        check(lib().qpsk_demod_constellation(self._h, _ptr(x), n, _ptr(y), cap, _ptr(ns)))
        outs = [y[c, : 2 * ns[c]].copy() for c in range(self.channels)]
        return outs[0] if self.channels == 1 else outs

    def bits_bound(self, n_floats: int) -> int:
        b = C.c_int64(0)
        check(lib().qpsk_demod_bits_bound(self._h, n_floats, C.byref(b)))
        return b.value

    def demod_bits_dev(self, d_in: int, n_floats: int, in_stride: int, d_bits: int, bits_cap: int, d_n_bits: int, stream: int = 0):
        check(lib().qpsk_demod_bits_dev(self._h, d_in, n_floats, in_stride or n_floats, d_bits, bits_cap, d_n_bits, stream))

    def demod_bytes_dev(self, d_in: int, n_floats: int, in_stride: int, startMarker: bytes, endMarker: bytes, d_payload: int,
                        payload_cap: int, d_n_bytes: int, stream: int = 0):
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        check(lib().qpsk_demod_bytes_dev(self._h, d_in, n_floats, in_stride or n_floats, _ptr(s), s.size, _ptr(e), e.size,
                                         d_payload, payload_cap, d_n_bytes, stream))

    def loop_state(self):
        Cn = self.channels
        ct, cf, mu, mi = (np.empty(Cn, np.float64) for _ in range(4))
        fp, ff = np.empty(Cn, np.float32), np.empty(Cn, np.float32)
        check(lib().qpsk_demod_loop_state(self._h, ct.ctypes.data_as(N.f64p), cf.ctypes.data_as(N.f64p), mu.ctypes.data_as(N.f64p),
                                          mi.ctypes.data_as(N.f64p), fp.ctypes.data_as(N.f32p), ff.ctypes.data_as(N.f32p)))
        d = dict(costas_theta=ct, costas_freq=cf, mm_mu=mu, mm_integral=mi, fll_phase=fp, fll_freq=ff)
        return {k: (float(v[0]) if Cn == 1 else v) for k, v in d.items()}

    @property
    def in_frame(self):
        f = np.zeros(self.channels, np.int32)
        check(lib().qpsk_demod_in_frame(self._h, f.ctypes.data_as(N.i32p)))
        return bool(f[0]) if self.channels == 1 else f.astype(bool)


# ---- synthetic channel / BER (SURVEY 8f-1, K6, K7) ----------------------------------------------
class SimChannel(_Handle):
    """Two unstable LOs (TB/Simulated/LocalOscilator.cs) + AWGN (TB/HelperModels.cs) + static multipath."""
    _destroy = "qpsk_chan_destroy"

    def __init__(self, tx_freq_hz, rx_freq_hz, sample_rate_hz, tx_ppm=0.0, rx_ppm=0.0, tx_phase0=0.0, rx_phase0=0.0,
                 noise_dbfs=-1000.0, mode=0, path_gains_iq=(), path_delays=(), seed=0, channels=1, first_channel=0):
        super().__init__()
        self.channels = channels
        p = ChanParams()
        p.tx_freq_hz, p.rx_freq_hz, p.sample_rate_hz = tx_freq_hz, rx_freq_hz, sample_rate_hz
        p.tx_ppm, p.rx_ppm, p.tx_phase0, p.rx_phase0 = tx_ppm, rx_ppm, tx_phase0, rx_phase0
        p.noise_dbfs, p.mode, p.n_paths, p.seed = noise_dbfs, mode, len(path_delays), seed
        for k, d in enumerate(path_delays):
            p.path_delay[k] = int(d)
            p.path_gain_iq[2 * k] = float(path_gains_iq[2 * k])
            p.path_gain_iq[2 * k + 1] = float(path_gains_iq[2 * k + 1])
        check(lib().qpsk_chan_create(C.byref(p), channels, first_channel, C.byref(self._h)))

    def apply(self, x_iq) -> np.ndarray:
        x = _f32(x_iq)
        n = x.shape[-1] if x.ndim == 2 else x.size
        y = np.empty_like(x)
        check(lib().qpsk_chan_apply(self._h, _ptr(x), n, _ptr(y)))
        return y

    def apply_dev(self, d_x: int, n_floats: int, x_stride: int, d_y: int, y_stride: int, stream: int = 0):
        check(lib().qpsk_chan_apply_dev(self._h, d_x, n_floats, x_stride, d_y, y_stride, stream))


def fill_bytes_dev(seed: int, first_channel: int, channels: int, n_bytes: int, d_out: int, stream: int = 0):
    check(lib().qpsk_fill_bytes_dev(seed, first_channel, channels, n_bytes, d_out, stream))


def unpack_bits_dev(d_bytes: int, n_bytes: int, bytes_stride: int, channels: int, d_bits: int, bits_stride: int, stream: int = 0):
    check(lib().qpsk_unpack_bits_dev(d_bytes, n_bytes, bytes_stride, channels, d_bits, bits_stride, stream))


def pack_bits_dev(d_bits: int, bits_stride: int, d_n_bits: int, max_bits: int, channels: int, d_packed: int, packed_stride: int,
                  stream: int = 0):
    check(lib().qpsk_pack_bits_dev(d_bits, bits_stride, d_n_bits, max_bits, channels, d_packed, packed_stride, stream))


def ber_count_dev(d_rx_bits: int, rx_stride: int, d_n_rx: int, d_ref_bits: int, ref_stride: int, n_ref: int, channels: int,
                  d_counters: int, stream: int = 0):
    check(lib().qpsk_ber_count_dev(d_rx_bits, rx_stride, d_n_rx, d_ref_bits, ref_stride, n_ref, channels, d_counters, stream))


# ---- §8f-2: the full receive chain of TB/Simulated/testFullDemodChain.cs, repaired -----------------
class FullDemodChain(_Handle):
    """FLL -> RRC matched filter -> Mueller-Muller -> Costas as testFullDemodChain.cs:22-110 wires the blocks by hand,
    on the GPU over `channels` independent streams.  Defaults are the literal values of that test (:18-45); every
    block parameter can be overridden by keyword (the field names of qpsk_chain_params)."""
    _destroy = "qpsk_chain_destroy"
    TOPICS = ("baseband", "baseband_PostSymbolSync", "baseband_PostSymbolSyncPostCostas")   # :95, :103, :110

    def __init__(self, channels: int = 1, **overrides):
        super().__init__()
        self.channels = channels
        p = N.ChainParams()
        check(lib().qpsk_chain_default_params(C.byref(p)))
        names = {f[0] for f in N.ChainParams._fields_}
        for k, v in overrides.items():
            if k not in names:
                raise TypeError(f"unknown chain parameter {k!r}")
            setattr(p, k, v)
        self.params = p
        check(lib().qpsk_chain_create(C.byref(p), channels, C.byref(self._h)))

    def set_fir_mode(self, mode: int):
        check(lib().qpsk_chain_set_fir_mode(self._h, mode))

    def symbols_bound(self, n_floats: int) -> int:
        b = C.c_int64(0)
        check(lib().qpsk_chain_symbols_bound(self._h, n_floats, C.byref(b)))
        return b.value

    def Process(self, samplesIQ):
        """-> (baseband, post_symbol_sync, post_costas): float32 interleaved IQ arrays (lists of per-channel arrays for
        batch handles) — the payloads of the three ZMQ topics of one loop pass."""
        if samplesIQ is None:
            raise ArgumentNullException("samplesIQ")
        x = _f32(samplesIQ)
        n = x.shape[-1] if x.ndim == 2 else x.size
        cap = max(self.symbols_bound(n), 2) if n % 2 == 0 else 2
        bb = np.zeros((self.channels, n), np.float32)
        sy = np.zeros((self.channels, cap), np.float32)
        co = np.zeros((self.channels, cap), np.float32)
        ns = np.zeros(self.channels, np.int32)
        check(lib().qpsk_chain_process(self._h, _ptr(x), n, _ptr(bb), _ptr(sy), _ptr(co), cap, ns.ctypes.data_as(N.i32p)))
        if self.channels == 1:
            return bb[0], sy[0, : 2 * ns[0]].copy(), co[0, : 2 * ns[0]].copy()
        return ([bb[c] for c in range(self.channels)], [sy[c, : 2 * ns[c]].copy() for c in range(self.channels)],
                [co[c, : 2 * ns[c]].copy() for c in range(self.channels)])

    def zmq_frames(self, samplesIQ, frame_samples: int = 4096):
        """The multipart messages testFullDemodChain.cs:88-110 publishes for this input, in order: per
        `frame_samples` block one ("baseband", bytes) message and, when the block produced symbols, the two symbol
        topics.  Payloads are raw little-endian cf32 (Buffer.BlockCopy of the float arrays), what the GNU Radio
        ZMQ SUB sources of the viewers read.  Single-channel handles only."""
        if self.channels != 1:
            raise N.ArgumentException("zmq_frames is per stream; use Process on batch handles")
        x = _f32(samplesIQ)
        out = []
        step = 2 * frame_samples
        for a in range(0, x.size, step):
            bb, sy, co = self.Process(x[a:a + step])
            out.append((self.TOPICS[0].encode(), bb.astype("<f4").tobytes()))
            if sy.size:                                              # `if (decided.Length > 0)` :97
                out.append((self.TOPICS[1].encode(), sy.astype("<f4").tobytes()))
                out.append((self.TOPICS[2].encode(), co.astype("<f4").tobytes()))
        return out

    def process_dev(self, d_in: int, n_floats: int, in_stride: int, d_baseband: int, bb_stride: int, d_sync: int,
                    sync_stride: int, d_costas: int, costas_stride: int, d_n_sym: int, stream: int = 0):
        check(lib().qpsk_chain_process_dev(self._h, d_in, n_floats, in_stride or n_floats, d_baseband, bb_stride or n_floats,
                                           d_sync, sync_stride, d_costas, costas_stride, d_n_sym, stream))

    def loop_state(self):
        Cn = self.channels
        fp, ff = np.empty(Cn, np.float32), np.empty(Cn, np.float32)
        mu, ct, cf = (np.empty(Cn, np.float64) for _ in range(3))
        check(lib().qpsk_chain_loop_state(self._h, fp.ctypes.data_as(N.f32p), ff.ctypes.data_as(N.f32p), mu.ctypes.data_as(N.f64p),
                                          ct.ctypes.data_as(N.f64p), cf.ctypes.data_as(N.f64p)))
        d = dict(fll_phase=fp, fll_freq=ff, mm_mu=mu, costas_theta=ct, costas_freq=cf)
        return {k: (float(v[0]) if Cn == 1 else v) for k, v in d.items()}


# ---- §8f-3: streaming front-end + CS16 -----------------------------------------------------------
class StreamingDemodulator(_Handle):
    """The receive loop of TB/SDR/ModDemodOverSDR.cs:116-183 without the per-block wait: push() a block (one radio
    MTU), poll() payloads in push order.  Block k's payload is what the k-th DeModulateBytes(block, start, end) call
    returns on the same QPSKDeModulator."""
    _destroy = "qpsk_stream_destroy"

    def __init__(self, demod: "QPSKDeModulator", startMarker: bytes, endMarker: bytes, max_block_floats: int,
                 max_payload_bytes: int = 1 << 16, depth: int = 4):
        super().__init__()
        self.demod = demod                       # keeps the demodulator alive
        self.max_payload = max_payload_bytes
        s, e = _bytes_arr(startMarker), _bytes_arr(endMarker)
        check(lib().qpsk_stream_create(demod._h, max_block_floats, max_payload_bytes, depth, _ptr(s), s.size, _ptr(e), e.size,
                                       C.byref(self._h)))
        self._buf = np.empty(max_payload_bytes, np.uint8)

    def push(self, samplesIQ):
        x = _f32(samplesIQ)
        check(lib().qpsk_stream_push(self._h, _ptr(x), x.size))

    def push_cs16(self, samplesI16, scale: float = 1.0 / 32768.0):
        x = np.ascontiguousarray(samplesI16, np.int16)
        check(lib().qpsk_stream_push_cs16(self._h, _ptr(x), x.size, scale))

    def poll(self, wait: bool = False):
        """-> payload bytes of the next finished block (b"" when it held no complete frame), or None when no block
        is ready."""
        n, have = C.c_int64(0), C.c_int(0)
        check(lib().qpsk_stream_poll(self._h, int(wait), _ptr(self._buf), self._buf.size, C.byref(n), C.byref(have)))
        if not have.value:
            return None
        return self._buf[: n.value].tobytes()

    def pending(self):
        a, b = C.c_int64(0), C.c_int64(0)
        check(lib().qpsk_stream_pending(self._h, C.byref(a), C.byref(b)))
        return a.value - b.value

    def flush(self):
        check(lib().qpsk_stream_flush(self._h))

    def drain(self):
        """Wait for every pushed block and return their payloads in order."""
        out = []
        while self.pending():
            out.append(self.poll(wait=True))
        return out

    def close(self):
        super().close()
        self.demod = None


def SaveAsCs16(iq) -> tuple:
    """HelperFunctions.SaveAsCs16 (MS/Models/HelperFunctions.cs:75-106) without the file: -> (int16 array, maxVal)."""
    x = _f32(iq)
    out = np.empty(x.size, np.int16)
    m = C.c_float(0)
    check(lib().qpsk_cf32_to_cs16(_ptr(x), x.size, _ptr(out), C.byref(m)))
    return out, m.value


def Cs16ToCf32(iq16, scale: float = 1.0 / 32768.0) -> np.ndarray:
    x = np.ascontiguousarray(iq16, np.int16)
    out = np.empty(x.size, np.float32)
    check(lib().qpsk_cs16_to_cf32(_ptr(x), x.size, scale, _ptr(out)))
    return out
