"""fp64 CPU restatements of the digital down-converter bank (include/qpskcuda.h, "digital down-converter bank").
Test infrastructure only: the library never imports this.

- phase_word: inc = nearbyint(ldexp(f, 64)) mod 2^64, as a Python int.
- ddc_direct: the definition taken literally: mix every sample down by its own phase word, filter with h, keep n_m = mD + D-1.
- DdcPoly: the rotated-tap form the kernel computes, streaming (history, pending samples and the 64-bit counter kept
  across calls); `start` begins the counter elsewhere than 0 (with a zero history), to check phases past 2^32 samples.
- ddc_scene: a wideband capture of QPSK carriers at arbitrary frequencies, built with the same phase words.
"""
from __future__ import annotations

import numpy as np
from scipy.signal import fftconvolve, firwin, kaiser_beta

TWO64 = 2.0 ** 64


def phase_word(f: float) -> int:
    return int(np.rint(np.ldexp(np.float64(f), 64))) % (1 << 64)


def phase_angle(inc: int, n) -> np.ndarray:
    """2 pi phi(n) / 2^64 in (-pi, pi], phi(n) = inc * n mod 2^64, for an array of stream indices n >= 0."""
    phi = np.uint64(inc) * np.asarray(n, dtype=np.uint64)           # numpy uint64 products wrap mod 2^64
    return 2 * np.pi * (phi.view(np.int64).astype(np.float64) / TWO64)


def ddc_direct(h, freqs, D: int, x) -> np.ndarray:
    """y[k, m] = sum_i h[i] x[n_m - i] e^{-j 2 pi phi_k(n_m - i) / 2^64}, n_m = mD + D-1, over the outputs x completes."""
    h = np.asarray(h, np.float64)
    x = np.asarray(x, np.complex128)
    n_out = x.size // D
    keep = np.arange(n_out) * D + D - 1
    n = np.arange(x.size)
    y = np.empty((len(freqs), n_out), np.complex128)
    with np.errstate(over="ignore"):
        for k, f in enumerate(freqs):
            mixed = x * np.exp(-1j * phase_angle(phase_word(f), n))
            y[k] = np.convolve(mixed, h)[keep]
    return y


class DdcPoly:
    """u_k[m] = sum_i g_k[i] x[n_m - i], g_k[i] = h[i] e^{+j 2 pi phi_k(i) / 2^64}, y_k[m] = u_k[m] e^{-j 2 pi phi_k(n_m) / 2^64},
    over a stream fed in any chunks.  Keeps the last N-1 samples, the pending samples of the open block and the counter."""

    def __init__(self, h, freqs, D: int, start: int = 0):
        self.h = np.asarray(h, np.float64)
        self.D = D
        self.N = self.h.size
        self.inc = [phase_word(f) for f in freqs]
        i = np.arange(self.N)
        with np.errstate(over="ignore"):
            self.G = np.array([self.h * np.exp(1j * phase_angle(c, i)) for c in self.inc])     # [K, N]
        self.start = start
        self.reset()

    def reset(self):
        self.count = self.start
        self.buf = np.zeros(self.N - 1 + self.count % self.D, np.complex128)

    def process(self, x) -> np.ndarray:
        D, N = self.D, self.N
        x = np.asarray(x, np.complex128).ravel()
        pending = self.count % D
        z = np.concatenate([self.buf, x])
        n_out = (pending + x.size) // D
        y = np.empty((len(self.inc), n_out), np.complex128)
        base = self.count - pending + D - 1                          # n_m of this call's first output
        step = max(1, (1 << 22) // max(N, 1))
        for j0 in range(0, n_out, step):                            # windows W[j, i] = z[jD + D-1 + N-1 - i]
            j = np.arange(j0, min(n_out, j0 + step))
            W = z[(j * D + D - 1 + N - 1)[:, None] - np.arange(N)[None, :]]
            u = self.G @ W.T
            n_m = (np.uint64(base % (1 << 64)) + j.astype(np.uint64) * np.uint64(D))
            with np.errstate(over="ignore"):
                rot = np.array([np.exp(-1j * phase_angle(c, n_m)) for c in self.inc])
            y[:, j0:j0 + j.size] = u * rot
        self.buf = z[n_out * D:]
        self.count += x.size
        return y


TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"
SCENE_FS, SCENE_RS = 4000, 1000           # channel rate and symbol rate: 4 samples per symbol at fs/D
SCENE_D, SCENE_P = 16, 8                  # decimation, prototype length P*D
# six carriers at uneven spacing, none on a k/16 grid point except 0.125, where the PFB would rotate channel 2 by 45 degrees
SCENE_FREQS = [-0.437, -0.3, -0.1709, 0.0219, 0.125, 0.2811]


def scene_taps(D: int = SCENE_D, P: int = SCENE_P) -> np.ndarray:
    """Kaiser-windowed lowpass, unit DC gain, P*D taps, cutoff 0.5/D cycles per sample, 60 dB."""
    return firwin(P * D, 1.0 / D, window=("kaiser", kaiser_beta(60.0)), scale=True)


def ddc_scene(orc, h, D: int, freqs, seed: int, n_payload: int = 48):
    """A wideband capture with one QPSK frame (oracle.QPSKModulator, START/END markers, TSC) per frequency at channel rate
    SCENE_FS: each is upsampled by D (zeros stuffed), filtered with D*h, mixed up by e^{+j 2 pi phi_k(n) / 2^64} with the
    bank's own phase words, and the carriers are summed, plus complex AWGN of power 1e-4.  With h of N = P*D taps the
    interpolation and the bank's filter together delay a carrier by N-1 wide samples, so bank output m carries channel
    sample m - (P-1); each carrier has 41 leading zeros, so with P = 8 its burst starts on a symbol boundary of the
    demodulator's clock recovery, as an unpadded burst does.  Returns (wideband complex128, [payload per frequency])."""
    h = np.asarray(h, np.float64)
    rng = np.random.default_rng(seed)
    pays = [rng.integers(0, 256, n_payload, dtype=np.uint8).tobytes() for _ in freqs]
    mod = orc.QPSKModulator(SCENE_FS, SCENE_RS, 0.35, 10, True, TSC)
    car = []
    for p in pays:
        f = mod.ModulateBytes(p, b"START", b"END")
        car.append(np.concatenate([np.zeros(41), f[0::2].astype(np.float64) + 1j * f[1::2], np.zeros(80)]))
    n = max(c.size for c in car) * D
    t = np.arange(n)
    wide = np.zeros(n, np.complex128)
    with np.errstate(over="ignore"):
        for c, f in zip(car, freqs):
            up = np.zeros(n, np.complex128)
            up[: c.size * D: D] = c
            wide += fftconvolve(up, D * h)[:n] * np.exp(1j * phase_angle(phase_word(f), t))
    wide = wide + (rng.standard_normal(n) + 1j * rng.standard_normal(n)) * np.sqrt(1e-4 / 2)
    return wide, pays
