"""fp64 CPU restatements of the rational resampler (include/qpskcuda.h, "rational resampler").
Test infrastructure only: the library never imports this.

- resamp_count: outputs complete after n inputs, n == 0 ? 0 : floor((nL - 1) / M) + 1 (Python ints: no overflow).
- resamp_direct: the definition taken literally: zero-stuff by L, filter with h, keep every M-th sample.
- ResampPoly: the polyphase form the kernel computes, streaming over a [channels, n] batch (the last P-1 samples and the
  input / output counters kept across calls); `start` begins the input counter elsewhere than 0 (with a zero history),
  to check positions past 2^32 samples.
- check_params: the C limits, restated.
- resamp_scene: a wideband capture whose DDC output is not an integer number of samples per symbol.
"""
from __future__ import annotations

import numpy as np

MAX_TAPS, MAX_FACTOR, MAX_BRANCH, MAX_CHANNELS = 16384, 1024, 64, 16384
OK, ERR_ARG, ERR_UNSUPPORTED = "ok", "arg", "unsupported"


def resamp_count(n: int, L: int, M: int) -> int:
    return 0 if n == 0 else (n * L - 1) // M + 1


def branch_taps(N: int, L: int) -> int:
    return -(-N // L)


def check_params(n_taps: int, L: int, M: int, channels: int) -> str:
    """What qpsk_resamp_create returns for finite taps."""
    if n_taps <= 0:
        return ERR_ARG
    if (n_taps > MAX_TAPS or not 1 <= L <= MAX_FACTOR or not 1 <= M <= MAX_FACTOR or not 1 <= channels <= MAX_CHANNELS
            or branch_taps(n_taps, L) > MAX_BRANCH):
        return ERR_UNSUPPORTED
    return OK


def resamp_direct(h, L: int, M: int, x) -> np.ndarray:
    """y[m] = sum_i h[i] x_up[mM - i] over the outputs x completes (x: one row, or [channels, n])."""
    h = np.asarray(h, np.float64)
    x = np.asarray(x, np.complex128)
    if x.ndim == 2:
        return np.array([resamp_direct(h, L, M, r) for r in x]).reshape(x.shape[0], -1)
    up = np.zeros(x.size * L, np.complex128)
    up[::L] = x
    n_out = resamp_count(x.size, L, M)
    full = np.convolve(up, h)
    return full[np.arange(n_out) * M]


class ResampPoly:
    """y[m] = sum_q h[phi_m + qL] x[n_m - q], n_m = floor(mM / L), phi_m = mM mod L, over a [channels, n] stream fed in any
    chunks.  Keeps the last P-1 samples of each channel and the input and output counters."""

    def __init__(self, h, L: int, M: int, channels: int = 1, start: int = 0):
        h = np.asarray(h, np.float64).ravel()
        self.L, self.M, self.C = L, M, channels
        self.P = branch_taps(h.size, L)
        hp = np.zeros(self.P * L)
        hp[: h.size] = h
        self.hT = hp.reshape(self.P, L).T.copy()                   # [L][P]: hT[phi][q] = h[phi + qL]
        self.start = start
        self.reset()

    def reset(self):
        self.n_in = self.start
        self.n_outc = resamp_count(self.start, self.L, self.M)
        self.hist = np.zeros((self.C, self.P - 1), np.complex128)

    def outputs_for(self, n: int) -> int:
        return resamp_count(self.n_in + n, self.L, self.M) - self.n_outc

    def process(self, x) -> np.ndarray:
        x = np.asarray(x, np.complex128).reshape(self.C, -1)
        L, M, P = self.L, self.M, self.P
        z = np.concatenate([self.hist, x], axis=1)
        n_out = self.outputs_for(x.shape[1])
        m = self.n_outc + np.arange(n_out, dtype=object)
        n_m = np.array([int(v) * M // L for v in m], dtype=np.int64) if n_out else np.zeros(0, np.int64)
        phi = np.array([int(v) * M % L for v in m], dtype=np.int64) if n_out else np.zeros(0, np.int64)
        d = n_m - self.n_in                                        # into z: tap q reads z[d + P-1 - q]
        y = np.zeros((self.C, n_out), np.complex128)
        step = max(1, (1 << 22) // max(P * self.C, 1))
        for a in range(0, n_out, step):
            sl = slice(a, min(n_out, a + step))
            idx = (d[sl] + P - 1)[:, None] - np.arange(P)[None, :]   # [t, q]
            taps = self.hT[phi[sl]]                                  # [t, q]
            y[:, sl] = np.einsum("tq,ctq->ct", taps, z[:, idx])
        if P > 1:
            self.hist = z[:, z.shape[1] - (P - 1):]
        self.n_in += x.shape[1]
        self.n_outc += n_out
        return y


# ---- an end-to-end scene: carriers whose DDC output rate is not a multiple of the symbol rate ---------------------------
SCENE_FS, SCENE_RS = 4096, 1000           # DDC output rate and symbol rate: 4.096 samples per symbol
SCENE_L, SCENE_M = 125, 128               # 4096 * 125 / 128 = 4000 S/s: 4 samples per symbol
SCENE_D = 16
SCENE_FREQS = [-0.3, -0.1709, 0.0219, 0.2811]
LEAD_IN = 250                             # random bytes before START: the burst need not start on a symbol boundary


def resamp_taps(L: int, M: int, P: int = 24, atten: float = 60.0) -> np.ndarray:
    """L * Kaiser lowpass (unit DC gain per branch on average), P*L taps, cutoff at the narrower of the two Nyquist rates."""
    from scipy.signal import firwin, kaiser_beta
    return L * firwin(P * L, 0.9 / max(L, M), window=("kaiser", kaiser_beta(atten)), scale=True)


def resamp_scene(orc, tsc, seed: int, freqs=SCENE_FREQS, D: int = SCENE_D, n_payload: int = 40, lead_zeros: int = 2):
    """A wideband capture at D * SCENE_FS with one QPSK frame per frequency: each burst (oracle.QPSKModulator at 4 sps after
    a LEAD_IN-byte random lead-in before START) is resampled by 128/125 to 4.096 sps, upsampled by D with an ideal-ish
    lowpass and mixed up to its frequency; plus complex AWGN of power 1e-4.  `lead_zeros` 4-sps zeros go before each
    burst: the demodulator's burst-start acquisition depends on where the burst falls within a symbol (on the oracle
    demodulator, 0 / 1 / 4 / 5 zeros lose every frame of this scene after the resampler, 2 / 3 / 6 / 7 decode them all), so
    the scene is pinned at one alignment that decodes.  Returns (wideband complex128,
    [payload per frequency])."""
    from scipy.signal import fftconvolve, firwin, kaiser_beta, resample_poly
    from ddc_oracle import phase_angle, phase_word
    rng = np.random.default_rng(seed)
    pays = [rng.integers(0, 256, n_payload, dtype=np.uint8).tobytes() for _ in freqs]
    mod = orc.QPSKModulator(4000, SCENE_RS, 0.35, 10, True, tsc)
    car = []
    for p in pays:
        lead = rng.integers(0, 256, LEAD_IN, dtype=np.uint8).tobytes()
        f = mod.ModulateBytes(p, lead + b"START", b"END")   # the demodulator hunts for START alone
        c = f[0::2].astype(np.float64) + 1j * f[1::2]
        car.append(resample_poly(np.concatenate([np.zeros(lead_zeros), c, np.zeros(400)]), SCENE_M, SCENE_L))
    n = max(c.size for c in car) * D
    t = np.arange(n)
    g = D * firwin(16 * D, 1.0 / D, window=("kaiser", kaiser_beta(60.0)), scale=True)
    wide = np.zeros(n, np.complex128)
    with np.errstate(over="ignore"):
        for c, f in zip(car, freqs):
            up = np.zeros(n, np.complex128)
            up[: c.size * D: D] = c
            wide += fftconvolve(up, g)[:n] * np.exp(1j * phase_angle(phase_word(f), t))
    wide = wide + (rng.standard_normal(n) + 1j * rng.standard_normal(n)) * np.sqrt(1e-4 / 2)
    return wide, pays
