"""CPU restatement of the frame synchronizer of csrc/fsync.cu (definition in include/qpskcuda.h, "frame synchronizer").

Written from the definition, not from the kernel: the GPU must be bit-identical to it.
  * pattern: the code bits c_0..c_{2P-1} of 32 zero bits and START, encoded from state 0 (fec_oracle.encode).
  * soft values: fec_oracle.soft_coherent / soft_differential, symbol k against symbol k-1 in differential mode.
  * M_r(p) = sum_i (c_{2i} ? 1 : -1) s0_r(p+i) + (c_{2i+1} ? 1 : -1) s1_r(p+i), s_r the soft values of y j^-r; coherent
    M = max over r (lowest r on ties), differential r = 0; E(p) = sum |s0| + |s1| over the window.
  * detection: the first searched p (from delta, or the last frame's p* + F) with E > 0 and 256 M >= rho E is p0; the frame
    is at p* = argmax M over [p0, p0 + P) (lowest p on ties); window [p* - delta, p* + F) derotated by j^-r*.  A frame is
    reported by the call after which symbols p* + F - 1 and p0 + 2P - 2 have both arrived.
The stream of every channel is kept whole, and each call searches it from where the last one stopped."""
import numpy as np

import fec_oracle as V

LEAD_BITS, TAIL_BITS = 32, 6        # QPSK_CODED_LEAD_BITS / QPSK_CODED_TAIL_BITS
RHO_DEFAULT = 144                   # QPSK_FSYNC_RHO_DEFAULT
INFO = np.dtype([("position", "<i8"), ("metric", "<i4"), ("energy", "<i4"), ("rotation", "<i4"), ("channel", "<i4")])


def pattern(start):
    """START bytes -> the 2P pattern bits (0/1)"""
    bits = np.concatenate([np.zeros(LEAD_BITS, np.uint8), np.unpackbits(np.frombuffer(bytes(start), np.uint8))])
    return V.encode(bits[None])[0][0]


def frame_symbols(n_start, payload_bytes, n_end):
    return LEAD_BITS + 8 * (n_start + payload_bytes + n_end) + TAIL_BITS


def soft(y, differential, scale):
    """y complex64 [C, n] -> int64 s0, s1 [C, n]; differential: symbol 0 has no predecessor and gets (0, 0)"""
    y = np.asarray(y, np.complex64)
    if not differential:
        return V.soft_coherent(y, scale)
    s0 = np.zeros(y.shape, np.int64)
    s1 = np.zeros(y.shape, np.int64)
    if y.shape[1] > 1:
        s0[:, 1:], s1[:, 1:] = V.soft_differential(y[:, 1:], y[:, :-1], scale)
    return s0, s1


def correlate(s0, s1, pat, differential):
    """-> M, rotation, E [C, n - P + 1] for every window that fits"""
    P = pat.size // 2
    a = np.where(pat[0::2] != 0, 1, -1)
    b = np.where(pat[1::2] != 0, 1, -1)
    L = s0.shape[1] - P + 1
    if L <= 0:
        z = np.zeros((s0.shape[0], 0), np.int64)
        return z, z, z
    X = np.zeros((s0.shape[0], L), np.int64)
    Y = np.zeros_like(X)
    E = np.zeros_like(X)
    e = np.abs(s0) + np.abs(s1)
    for i in range(P):
        w0, w1 = s0[:, i: i + L], s1[:, i: i + L]
        X += a[i] * w0 + b[i] * w1
        Y += a[i] * w1 - b[i] * w0
        E += e[:, i: i + L]
    if differential:
        return X, np.zeros_like(X), E
    cand = np.stack([X, Y, -X, -Y])                    # r = 0..3
    r = np.argmax(cand, axis=0)                        # first maximum: the lowest r on ties
    return np.take_along_axis(cand, r[None], 0)[0], r, E


def derotate(y, r):
    y = np.asarray(y, np.complex64)
    re, im = y.real.astype(np.float32), y.imag.astype(np.float32)
    out = np.empty_like(y)
    if r == 0:
        return y.copy()
    if r == 1:
        out.real, out.imag = im, -re
    elif r == 2:
        out.real, out.imag = -re, -im
    else:
        out.real, out.imag = -im, re
    return out


class FrameSync:
    """Streaming synchronizer over `channels`; process() takes complex64 rows and per-channel counts and returns, per
    channel, the list of (window, info) the call completes."""

    def __init__(self, channels=1, differential=True, start=b"START", payload_bytes=64, n_end=3, scale=None, rho=0):
        self.C, self.diff = channels, bool(differential)
        self.scale = np.float32(V.DEFAULT_SCALE[self.diff] if scale is None else scale)
        self.rho = rho or RHO_DEFAULT
        self.pat = pattern(start)
        self.P = self.pat.size // 2
        self.F = frame_symbols(len(start), payload_bytes, n_end)
        self.delta = 1 if self.diff else 0
        self.payload_bytes = payload_bytes
        self.reset()

    @property
    def window(self):
        return self.F + self.delta

    def reset(self):
        self.y = [np.zeros(0, np.complex64) for _ in range(self.C)]
        self.next = np.full(self.C, self.delta, np.int64)
        self.pending = [None] * self.C               # (p*, r*, M, E) of a frame found but not yet complete

    def process(self, sym, n_sym=None):
        sym = np.asarray(sym, np.complex64).reshape(self.C, -1)
        n_sym = (np.full(self.C, sym.shape[1], np.int64) if n_sym is None
                 else np.clip(np.broadcast_to(np.asarray(n_sym, np.int64), (self.C,)), 0, sym.shape[1]))
        for c in range(self.C):
            self.y[c] = np.concatenate([self.y[c], sym[c, : n_sym[c]]])
        n = np.array([v.size for v in self.y], np.int64)
        Y = np.zeros((self.C, max(int(n.max()), 1)), np.complex64)
        for c in range(self.C):
            Y[c, : n[c]] = self.y[c]
        s0, s1 = soft(Y, self.diff, self.scale)
        M, R, E = correlate(s0, s1, self.pat, self.diff)
        hit = (E > 0) & (256 * M >= self.rho * E)
        out = [[] for _ in range(self.C)]
        P, F = self.P, self.F
        for c in range(self.C):
            p, nc = int(self.next[c]), int(n[c])
            lim = nc - 2 * P + 2
            while True:
                if self.pending[c] is None:
                    if p >= lim:
                        break
                    h = np.nonzero(hit[c, p:lim])[0]
                    if h.size == 0:
                        p = lim
                        break
                    p0 = p + int(h[0])
                    k = p0 + int(np.argmax(M[c, p0: p0 + P]))
                    self.pending[c] = (k, int(R[c, k]), int(M[c, k]), int(E[c, k]))
                k, r, m, e = self.pending[c]
                if k + F > nc:
                    p = k
                    break
                w = derotate(self.y[c][k - self.delta: k + F], r)
                out[c].append((w, np.array((k, m, e, r, c), INFO)))
                self.pending[c] = None
                p = k + F
            self.next[c] = p
        return out


# ---- test streams --------------------------------------------------------------------------------------------------
def frame_bits(start, payload, end):
    raw = np.frombuffer(bytes(start) + bytes(payload) + bytes(end), np.uint8)
    return np.concatenate([np.zeros(LEAD_BITS, np.uint8), np.unpackbits(raw), np.zeros(TAIL_BITS, np.uint8)])


def stream(rng, start, payloads, end, gaps, differential, rot=0):
    """random coded pairs, then frame, random pairs, frame, ... -> (complex64 symbols, frame positions p*, frame bits).
    Differential: the first symbol is the reference, so pair k is symbol k + 1."""
    parts, pos, fbits, at = [], [], [], 0
    for g, pay in zip(gaps, payloads):
        parts.append(rng.integers(0, 2, 2 * g).astype(np.uint8))
        at += g
        b = frame_bits(start, pay, end)
        pos.append(at + (1 if differential else 0))
        parts.append(V.encode(b[None])[0][0])
        fbits.append(b)
        at += b.size
    parts.append(rng.integers(0, 2, 2 * gaps[-1]).astype(np.uint8) if len(gaps) > len(payloads) else np.zeros(0, np.uint8))
    y = V.qpsk_symbols(np.concatenate(parts)[None], differential)[0]
    return (y * np.complex64(1j ** rot)).astype(np.complex64), pos, fbits


def awgn(rng, y, esn0_db):
    sd = np.float32(np.sqrt(0.5 * 10 ** (-esn0_db / 10)))
    return (y + sd * (rng.standard_normal(y.shape) + 1j * rng.standard_normal(y.shape))).astype(np.complex64)
