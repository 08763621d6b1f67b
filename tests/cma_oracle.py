"""CPU restatements of the blind CMA equalizer and of the demodulator's equalizer stage — TEST INFRASTRUCTURE.

The equalizer is the project's own block (the reference has none); its arithmetic is fixed in include/qpskcuda.h.  Two
restatements of it live here and must agree bit for bit (tests/test_oracle_equalizer.py):
  * CmaScalar  — one channel, numpy.float32 scalars, the spec read line by line (small cases only);
  * CmaBatch   — float32 arrays over channels (ragged counts, the demodulator's one-time discard), fast enough to check
                 thousands of channels; every array operation rounds like the scalar one (elementwise, no FMA).
EqDemod is the oracle demodulator with the stage: it wires the CPU oracle's own blocks (oracle/: FLL, RRC matched filter,
Mueller-Muller, Costas, framer) exactly as the oracle's QPSKDeModulator does and puts CmaBatch between Mueller-Muller and
Costas.  With the stage off it must reproduce oracle.QPSKDeModulator bit for bit, which pins the wiring.
"""
from __future__ import annotations

import math

import numpy as np

f32 = np.float32
LANES = 8
MAX_TAPS = 64


class EqArgumentError(ValueError):
    """status code of the C ABI the same parameters get: -3 (QPSK_ERR_RANGE) or -7 (QPSK_ERR_UNSUPPORTED)"""

    def __init__(self, status: int):
        super().__init__(f"status {status}")
        self.status = status


def check_params(n_taps, mu, modulus):
    mu, modulus = f32(mu), f32(modulus)
    if not (math.isfinite(mu) and mu >= 0) or not (math.isfinite(modulus) and modulus > 0):
        raise EqArgumentError(-3)
    if not 1 <= n_taps <= MAX_TAPS:
        raise EqArgumentError(-7)


# ---- one channel, scalars ----------------------------------------------------------------------------------------------
class CmaScalar:
    def __init__(self, n_taps, mu, modulus=1.0):
        check_params(n_taps, mu, modulus)
        self.n, self.mu, self.r2 = int(n_taps), f32(mu), f32(modulus)
        self.reset()

    def reset(self):
        self.wr = [f32(0.0)] * self.n
        self.wi = [f32(0.0)] * self.n
        self.wr[(self.n - 1) // 2] = f32(1.0)
        self.hist = [(f32(0.0), f32(0.0))] * self.n      # hist[k] = x_{n-k}

    @property
    def taps(self):
        t = np.empty(2 * self.n, np.float32)
        t[0::2], t[1::2] = self.wr, self.wi
        return t

    def process1(self, xr, xi):
        self.hist = [(f32(xr), f32(xi))] + self.hist[:-1]
        lane_r = [f32(0.0)] * LANES
        lane_i = [f32(0.0)] * LANES
        for k, (vr, vi) in enumerate(self.hist):
            lane_r[k % LANES] = lane_r[k % LANES] + (self.wr[k] * vr - self.wi[k] * vi)
            lane_i[k % LANES] = lane_i[k % LANES] + (self.wr[k] * vi + self.wi[k] * vr)

        def tree(s):
            return ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]))
        yr, yi = tree(lane_r), tree(lane_i)
        d = (yr * yr + yi * yi) - self.r2
        er = np.fmin(np.fmax(yr * d, f32(-1.0)), f32(1.0))     # fminf / fmaxf: a NaN operand yields the other one
        ei = np.fmin(np.fmax(yi * d, f32(-1.0)), f32(1.0))
        for k, (vr, vi) in enumerate(self.hist):
            self.wr[k] = self.wr[k] - self.mu * (er * vr + ei * vi)
            self.wi[k] = self.wi[k] - self.mu * (ei * vr - er * vi)
        return yr, yi

    def Process(self, iq):
        x = np.asarray(iq, np.float32)
        y = np.empty_like(x)
        for s in range(0, x.size, 2):
            y[s], y[s + 1] = self.process1(x[s], x[s + 1])
        return y


# ---- channels as array rows ----------------------------------------------------------------------------------------------
class CmaBatch:
    def __init__(self, n_taps, mu, modulus=1.0, channels=1):
        check_params(n_taps, mu, modulus)
        self.n, self.mu, self.r2, self.C = int(n_taps), f32(mu), f32(modulus), int(channels)
        self.reset()

    def reset(self):
        C, N = self.C, self.n
        self.wr = np.zeros((C, N), np.float32)
        self.wi = np.zeros((C, N), np.float32)
        self.wr[:, (N - 1) // 2] = 1.0
        self.vr = np.zeros((C, N), np.float32)       # v[:, k] = x_{n-k}
        self.vi = np.zeros((C, N), np.float32)
        self.drop = np.full(C, (N - 1) // 2, np.int64)

    @property
    def taps(self) -> np.ndarray:
        t = np.empty((self.C, 2 * self.n), np.float32)
        t[:, 0::2], t[:, 1::2] = self.wr, self.wi
        return t

    @taps.setter
    def taps(self, t):
        t = np.asarray(t, np.float32).reshape(self.C, 2 * self.n)
        self.wr, self.wi = t[:, 0::2].copy(), t[:, 1::2].copy()

    def process(self, x, lengths=None, drop=False):
        """x [C, 2L] interleaved; channel c takes lengths[c] symbols (default L).  -> list of per-channel outputs; with
        `drop` the first outputs of the stream (the group delay, once) are discarded."""
        x = np.asarray(x, np.float32).reshape(self.C, -1)
        n = np.full(self.C, x.shape[1] // 2, np.int64) if lengths is None else np.asarray(lengths, np.int64)
        T = int(n.max()) if self.C else 0
        yr_all = np.zeros((self.C, T), np.float32)
        yi_all = np.zeros((self.C, T), np.float32)
        m1, p1, mu, r2 = f32(-1.0), f32(1.0), self.mu, self.r2
        N = self.n
        for t in range(T):
            act = t < n
            a2 = act[:, None]
            xr = np.where(act, x[:, 2 * t] if 2 * t < x.shape[1] else f32(0), f32(0)).astype(np.float32)
            xi = np.where(act, x[:, 2 * t + 1] if 2 * t < x.shape[1] else f32(0), f32(0)).astype(np.float32)
            vr = np.where(a2, np.concatenate([xr[:, None], self.vr[:, :-1]], axis=1), self.vr)
            vi = np.where(a2, np.concatenate([xi[:, None], self.vi[:, :-1]], axis=1), self.vi)
            pr = self.wr * vr - self.wi * vi
            pi = self.wr * vi + self.wi * vr
            sr = np.zeros((self.C, LANES), np.float32)
            si = np.zeros((self.C, LANES), np.float32)
            for j in range(0, N, LANES):
                w = min(LANES, N - j)
                sr[:, :w] = sr[:, :w] + pr[:, j:j + w]
                si[:, :w] = si[:, :w] + pi[:, j:j + w]
            yr = ((sr[:, 0] + sr[:, 1]) + (sr[:, 2] + sr[:, 3])) + ((sr[:, 4] + sr[:, 5]) + (sr[:, 6] + sr[:, 7]))
            yi = ((si[:, 0] + si[:, 1]) + (si[:, 2] + si[:, 3])) + ((si[:, 4] + si[:, 5]) + (si[:, 6] + si[:, 7]))
            d = (yr * yr + yi * yi) - r2
            er = np.fmin(np.fmax(yr * d, m1), p1)[:, None]
            ei = np.fmin(np.fmax(yi * d, m1), p1)[:, None]
            gr = er * vr + ei * vi
            gi = ei * vr - er * vi
            self.wr = np.where(a2, self.wr - mu * gr, self.wr)
            self.wi = np.where(a2, self.wi - mu * gi, self.wi)
            self.vr, self.vi = vr, vi
            yr_all[:, t], yi_all[:, t] = yr, yi
        out = []
        for c in range(self.C):
            k = int(n[c])
            dc = min(int(self.drop[c]), k) if drop else 0
            if drop:
                self.drop[c] -= dc
            y = np.empty(2 * (k - dc), np.float32)
            y[0::2], y[1::2] = yr_all[c, dc:k], yi_all[c, dc:k]
            out.append(y)
        return out


# ---- the oracle demodulator with the stage ------------------------------------------------------------------------------
class EqDemod:
    """`channels` copies of oracle.QPSKDeModulator(fs, rs, alpha, span, tsc=..., use_fll=...) with the library's equalizer
    stage: FLL? -> RRC matched filter -> Mueller-Muller -> [CMA, its first (N-1)//2 outputs discarded once] -> Costas ->
    decision -> (differential) bits -> TSC strip; DeModulateBytes hands the bits to the oracle's own framer."""

    def __init__(self, orc, fs, rs, alpha, span, channels=1, tsc=None, use_fll=False, diff=True, sym_bw=0.0001,
                 costas_bw=120.0, cfo_bw=float(np.float32(0.0001))):
        self.orc, self.C, self.tsc, self.use_fll, self.diff = orc, channels, tsc, use_fll, diff
        taps = orc.real_taps_to_iq(orc.RRCFilter.generateCoefficents(span, alpha, fs, rs))
        kp, ki = orc.mm_gains_from_bw(sym_bw)
        self.fll = [orc.FLLBandEdgeFilter(float(np.float32(fs // rs)), alpha, 40, float(np.float32(cfo_bw))) for _ in range(channels)]
        self.rrc = [orc.ComplexFIRFilter(taps) for _ in range(channels)]
        self.mm = [orc.MuellerMuller(fs / rs, kp, ki) for _ in range(channels)]
        self.costas = [orc.CostasLoopQpsk(float(rs), rs / costas_bw, 0.707) for _ in range(channels)]
        self.framer = [orc.QPSKDeModulator(fs, rs, alpha, span, tsc=tsc, use_fll=use_fll) for _ in range(channels)]
        self.have_prev = [False] * channels
        self.prev = [(f32(0), f32(0))] * channels
        self.eq = None

    def set_equalizer(self, n_taps, mu, modulus=1.0):
        if n_taps != 0:
            check_params(n_taps, mu, modulus)
        self.eq = CmaBatch(n_taps, mu, modulus, self.C) if n_taps else None

    def equalizer_taps(self):
        return self.eq.taps

    def _symbols(self, rx):
        rx = np.asarray(rx, np.float32).reshape(self.C, -1)
        syms = []
        for c in range(self.C):
            x = rx[c]
            if self.use_fll:
                x = self.fll[c].Process(x)
            syms.append(self.mm[c].Process(self.rrc[c].Filter(x)))
        if self.eq is None:
            return syms
        L = max(s.size for s in syms) if syms else 0
        pad = np.zeros((self.C, max(L, 2)), np.float32)
        for c, s in enumerate(syms):
            pad[c, : s.size] = s
        return self.eq.process(pad, [s.size // 2 for s in syms], drop=True)

    def deModulateConstellation(self, rx):
        return [self.costas[c].Process(s) for c, s in enumerate(self._symbols(rx))]

    def DeModulate(self, rx):
        rx = np.asarray(rx, np.float32).reshape(self.C, -1)
        if rx.shape[1] == 0:
            return [""] * self.C
        out = []
        for c, s in enumerate(self._symbols(rx)):
            y = self.costas[c].Process(s)
            dI = np.where(y[0::2] >= 0, f32(1.0), f32(-1.0)).astype(np.float32)
            dQ = np.where(y[1::2] >= 0, f32(1.0), f32(-1.0)).astype(np.float32)
            if self.diff:
                if dI.size and not self.have_prev[c]:
                    self.prev[c], self.have_prev[c] = (dI[0], dQ[0]), True
                    dI, dQ = dI[1:], dQ[1:]
                pI = np.concatenate([[self.prev[c][0]], dI[:-1]]).astype(np.float32)
                pQ = np.concatenate([[self.prev[c][1]], dQ[:-1]]).astype(np.float32)
                if dI.size:
                    self.prev[c] = (dI[-1], dQ[-1])
                delI = dI * pI + dQ * pQ
                delQ = dQ * pI - dI * pQ
                b0 = np.where(np.abs(delI) >= np.abs(delQ), delI < 0, delQ < 0)
                b1 = np.where(np.abs(delI) >= np.abs(delQ), delI < 0, delQ >= 0)
            else:
                b0, b1 = dI >= 0, dQ >= 0                     # "00" / "01" for dI < 0, "10" / "11" otherwise
            bits = np.empty(2 * b0.size, np.uint8)
            bits[0::2], bits[1::2] = b0, b1
            s_bits = (bits + ord("0")).tobytes().decode("ascii")
            if self.tsc:
                i = s_bits.find(self.tsc)
                s_bits = "" if i < 0 else s_bits[i + len(self.tsc):]
            out.append(s_bits)
        return out

    def DeModulateBytes(self, rx, sm: bytes, em: bytes, cap: int = 1 << 16):
        return [self.framer[c].FrameBits(b, sm, em, cap=cap) for c, b in enumerate(self.DeModulate(rx))]
