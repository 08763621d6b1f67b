"""fp64 CPU restatements of the polyphase analysis channelizer (include/qpskcuda.h, "polyphase analysis channelizer").
Test infrastructure only: the library never imports this.

- pfb_direct: the definition taken literally, one bandpass filter per channel, output kept at n = mM + M - 1.
- PfbPoly: the polyphase form, streaming (history and pending samples kept across calls), DFT by np.fft.ifft(...) * M.
- fdm_synthesize: the matching synthesis side, per-channel baseband streams -> one wideband stream.
"""
from __future__ import annotations

import numpy as np
from scipy.signal import fftconvolve


def pfb_direct(h, M: int, x) -> np.ndarray:
    """y[k, m] = sum_i h[i] e^{+j 2 pi k i / M} x[mM + M-1 - i] over the complete blocks of x (x = 0 before the start)."""
    h = np.asarray(h, np.float64)
    x = np.asarray(x, np.complex128)
    n_out = x.size // M
    keep = np.arange(n_out) * M + M - 1
    y = np.empty((M, n_out), np.complex128)
    i = np.arange(h.size)
    for k in range(M):
        g = h * np.exp(2j * np.pi * ((k * i) % M) / M)          # exact argument reduction
        y[k] = np.convolve(x, g)[keep]
    return y


class PfbPoly:
    """The polyphase form v_r[m] = sum_q h[qM + r] x[(m-q)M + M-1-r], y[:, m] = ifft(v[m]) * M, over a stream fed in any
    chunks; keeps the last (P-1) complete blocks and the pending samples of the open block."""

    def __init__(self, h, M: int):
        h = np.asarray(h, np.float64)
        self.M = M
        self.P = -(-h.size // M)
        hp = np.zeros(self.P * M)
        hp[: h.size] = h
        self.H = hp.reshape(self.P, M)              # H[q, r] = h[qM + r]
        self.reset()

    def reset(self):
        self.buf = np.zeros((self.P - 1) * self.M, np.complex128)

    def process(self, x) -> np.ndarray:
        M, P = self.M, self.P
        z = np.concatenate([self.buf, np.asarray(x, np.complex128).ravel()])
        n_out = (z.size - (P - 1) * M) // M
        Zr = z[: (n_out + P - 1) * M].reshape(n_out + P - 1, M)[:, ::-1]   # Zr[j, r] = z[jM + M-1-r]
        v = np.zeros((n_out, M), np.complex128)
        for q in range(P):
            v += self.H[q] * Zr[P - 1 - q: P - 1 - q + n_out]
        self.buf = z[n_out * M:]
        return (np.fft.ifft(v, axis=1) * M).T.copy()


def fdm_synthesize(h, M: int, carriers: dict, n_out: int | None = None) -> np.ndarray:
    """Wideband stream from per-channel baseband streams {k: samples at rate 1/M}: each is upsampled by M (zeros
    stuffed), filtered with M*h and shifted to +k/M cycles per sample, and the channels are summed.  Through the
    analysis, channel k returns its carrier delayed by P-1 channel samples and times e^{-j 2 pi k / M}, up to the
    prototype's aliasing."""
    h = np.asarray(h, np.float64)
    n = max(len(c) for c in carriers.values()) * M if n_out is None else n_out
    t = np.arange(n)
    out = np.zeros(n, np.complex128)
    for k, c in carriers.items():
        up = np.zeros(n, np.complex128)
        c = np.asarray(c, np.complex128)[: -(-n // M)]
        up[: c.size * M: M] = c
        out += fftconvolve(up, M * h)[:n] * np.exp(2j * np.pi * k * t / M)
    return out


TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"
SCENE_FS, SCENE_RS = 4000, 1000           # channel rate and symbol rate: 4 samples per symbol at fs/M


def qpsk_fdm_scene(orc, h, M: int, occupied, seed: int, n_payload: int = 48):
    """A wideband capture with QPSK frames (oracle.QPSKModulator, START/END markers, TSC) on the `occupied` channels at
    channel rate SCENE_FS, synthesized by fdm_synthesize, plus complex AWGN of power 1e-4 (-40 dBFS for unit-power
    carriers).  Each carrier has 41 leading zeros: with the analysis delay of P-1 = 7 channel samples the burst starts on
    a symbol boundary of the demodulator's clock recovery, as an unpadded burst does.  Returns (wideband complex128,
    {k: payload})."""
    rng = np.random.default_rng(seed)
    pays = {k: rng.integers(0, 256, n_payload, dtype=np.uint8).tobytes() for k in occupied}
    mod = orc.QPSKModulator(SCENE_FS, SCENE_RS, 0.35, 10, True, TSC)
    car = {}
    for k in occupied:
        f = mod.ModulateBytes(pays[k], b"START", b"END")
        car[k] = np.concatenate([np.zeros(41), f[0::2].astype(np.float64) + 1j * f[1::2], np.zeros(80)])
    wide = fdm_synthesize(h, M, car)
    wide = wide + (rng.standard_normal(wide.size) + 1j * rng.standard_normal(wide.size)) * np.sqrt(1e-4 / 2)
    return wide, pays


def scene_channels(M: int, n: int):
    """n occupied channels of an M-channel scene, in groups around k = 0, M/4, M/2, 3M/4: the analysis rotates channel k
    by e^{-j 2 pi k / M}, and these keep that rotation within 22.5 degrees of a multiple of 90 degrees, away from the
    45-degree point where the demodulator's Costas loop starts on its unstable equilibrium."""
    per = n // 4
    return sorted((j * M // 4 + d) % M for j in range(4) for d in range(-(per // 2), per - per // 2))
