"""CPU restatements of the feed-forward AGC (include/qpskcuda.h, "feed-forward AGC").  Test infrastructure only: the
library never imports this.

Stream form, per channel, with z = (the last W-1 input samples, zero before the stream) ++ this call's samples:
    env(v) = fmaxf(|v.re|, |v.im|)
    m[i]   = fmaxf over {0, env(z[i]), ..., env(z[i+W-1])}        (a NaN envelope is ignored)
    g[i]   = fminf(ref / m[i], max_gain)                           (fp32; m = 0 gives max_gain)
    y[i]   = (z[i].re * g[i], z[i].im * g[i])                      (fp32)
so output i carries the oldest sample of its window: the stream comes out W-1 samples late (GNU Radio's
feedforward_agc_cc, made causal).  No operation rounds more than once, so the two forms below agree bit for bit.

- AgcScalar: the definition taken literally, one output at a time (small cases only).
- AgcBatch: numpy over [channels, n], the sliding maximum by van Herk / Gil-Werman block prefix and suffix maxima.
- AgcDemod: AgcBatch (its first W-1 outputs discarded once) in front of one oracle.QPSKDeModulator per channel.
"""
from __future__ import annotations

import numpy as np

f32 = np.float32
MAX_WINDOW = 4096


def check_params(window: int, ref: float, max_gain: float):
    """The C checks: window 1..4096 (else unsupported), ref and max_gain finite and > 0 (else out of range)."""
    if window < 1 or window > MAX_WINDOW:
        raise NotImplementedError(f"window {window} outside 1..{MAX_WINDOW}")
    for name, v in (("ref", ref), ("max_gain", max_gain)):
        if not (np.isfinite(f32(v)) and f32(v) > 0):
            raise ValueError(f"{name} must be finite and > 0")


def _split(x, channels):
    x = np.asarray(x)
    if not np.iscomplexobj(x):
        x = np.ascontiguousarray(x, np.float32).reshape(channels, -1).view(np.complex64)
    return np.ascontiguousarray(x, np.complex64).reshape(channels, -1)


class _AgcBase:
    def __init__(self, window: int, ref: float, max_gain: float, channels: int = 1):
        check_params(window, ref, max_gain)
        self.W, self.ref, self.max_gain, self.C = window, f32(ref), f32(max_gain), channels
        self.reset()

    def reset(self):
        self.hist = np.zeros((self.C, self.W - 1), np.complex64)
        self.gain = np.full(self.C, self.max_gain, np.float32)      # the gain the all-zero history gives

    def process(self, x) -> np.ndarray:
        """x: [channels, n] complex64 (or interleaved float32) -> [channels, n] complex64, state advanced."""
        x = _split(x, self.C)
        z = np.concatenate([self.hist, x], axis=1)
        n = x.shape[1]
        if n == 0:
            return x.copy()
        m = self._window_max(z, n)
        with np.errstate(divide="ignore", over="ignore"):
            g = np.minimum(self.ref / m, self.max_gain).astype(np.float32)
        zs = z[:, :n]
        y = np.empty((self.C, n), np.complex64)
        y.real = zs.real * g
        y.imag = zs.imag * g
        self.hist = z[:, n:].copy()
        self.gain = g[:, -1].copy()
        return y

    @staticmethod
    def env(z):
        return np.fmax(np.abs(z.real), np.abs(z.imag)).astype(np.float32)


class AgcScalar(_AgcBase):
    def _window_max(self, z, n):
        e = self.env(z)
        m = np.empty((self.C, n), np.float32)
        for c in range(self.C):
            for i in range(n):
                v = f32(0)
                for k in range(self.W):
                    v = np.fmax(v, e[c, i + k])
                m[c, i] = v
        return m


class AgcBatch(_AgcBase):
    def _window_max(self, z, n):
        """m[i] = max(S[i], P[i + W - 1]) over blocks of W: S the suffix maximum to the end of i's block, P the prefix maximum
        from the start of (i + W - 1)'s block; when i starts a block, S alone covers the window."""
        W = self.W
        e = self.env(z)
        nb = -(-(n + W - 1) // W)
        pad = np.zeros((self.C, nb * W), np.float32)
        pad[:, : e.shape[1]] = e
        blocks = pad.reshape(self.C, nb, W)
        P = np.fmax.accumulate(blocks, axis=2).reshape(self.C, -1)
        S = np.fmax.accumulate(blocks[:, :, ::-1], axis=2)[:, :, ::-1].reshape(self.C, -1)
        i = np.arange(n)
        m = np.fmax(S[:, i], np.where(i % W == 0, f32(0), P[:, i + W - 1]))
        return np.fmax(m, f32(0)).astype(np.float32)


class AgcDemod:
    """`channels` oracle.QPSKDeModulator(fs, rs, alpha, span, tsc=..., use_fll=...) behind the library's AGC stage: the
    AGC's first W-1 outputs of each stream are discarded once, so sample k reaching the FLL / matched filter is input
    sample k, scaled."""

    def __init__(self, orc, fs, rs, alpha, span, channels=1, tsc=None, use_fll=False):
        self.C = channels
        self.dem = [orc.QPSKDeModulator(fs, rs, alpha, span, tsc=tsc, use_fll=use_fll) for _ in range(channels)]
        self.agc = None
        self.drop = 0

    def set_agc(self, window: int, ref: float = 1.0, max_gain: float = 65536.0):
        if window == 0:
            self.agc = None
            return
        self.agc = AgcBatch(window, ref, max_gain, self.C)
        self.drop = window - 1

    def _rows(self, rx):
        x = _split(rx, self.C)
        if self.agc is not None:
            x = self.agc.process(x)
            dc = min(self.drop, x.shape[1])
            self.drop -= dc
            x = x[:, dc:]
        return [np.ascontiguousarray(r).view(np.float32) for r in x]

    def DeModulate(self, rx):
        return [d.DeModulate(r) for d, r in zip(self.dem, self._rows(rx))]

    def DeModulateBytes(self, rx, sm: bytes, em: bytes):
        return [d.DeModulateBytes(r, sm, em) for d, r in zip(self.dem, self._rows(rx))]
