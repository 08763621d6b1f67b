"""CPU restatements of the fractionally spaced (T/sps) blind CMA equalizer and of the demodulator's fractionally spaced
stage — TEST INFRASTRUCTURE.

The arithmetic is the symbol-spaced equalizer's (include/qpskcuda.h, restated in tests/cma_oracle.py) with an update stride
`sps`: every input sample shifts the window and forms and outputs y; the error and the tap update run only on stream samples
n with n % sps == 0, n a per-channel counter that persists across calls and resets to 0.  sps = 1 is the symbol-spaced
equalizer.  Two restatements, which must agree bit for bit (tests/test_oracle_fse.py):
  * FseScalar — one channel, numpy.float32 scalars, the spec read line by line (CmaScalar with the stride);
  * FseBatch  — float32 arrays over channels with the counter carried per channel (CmaBatch with the stride).
FseDemod is cma_oracle.EqDemod with the fractionally spaced stage: FLL? -> RRC matched filter -> [FseBatch(sps = fs/rs), its
first (N-1)//2 outputs discarded once] -> Mueller-Muller -> [CmaBatch] -> Costas -> decision -> bits.
"""
from __future__ import annotations

import numpy as np

from cma_oracle import LANES, CmaBatch, CmaScalar, EqArgumentError, EqDemod, check_params as check_eq_params

f32 = np.float32
MAX_SPS = 8


def check_params(n_taps, mu, modulus, sps):
    """the statuses of qpsk_eq_create_fractional: -3 for mu / modulus, then -7 for the tap count, then -7 for sps"""
    check_eq_params(n_taps, mu, modulus)
    if not 1 <= sps <= MAX_SPS:
        raise EqArgumentError(-7)


# ---- one channel, scalars ----------------------------------------------------------------------------------------------
class FseScalar(CmaScalar):
    def __init__(self, n_taps, mu, modulus=1.0, sps=1):
        check_params(n_taps, mu, modulus, sps)
        self.sps = int(sps)
        super().__init__(n_taps, mu, modulus)

    def reset(self):
        super().reset()
        self.count = 0                                  # stream sample counter n

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
        update = self.count % self.sps == 0
        self.count += 1
        if not update:
            return yr, yi
        d = (yr * yr + yi * yi) - self.r2
        er = np.fmin(np.fmax(yr * d, f32(-1.0)), f32(1.0))     # fminf / fmaxf: a NaN operand yields the other one
        ei = np.fmin(np.fmax(yi * d, f32(-1.0)), f32(1.0))
        for k, (vr, vi) in enumerate(self.hist):
            self.wr[k] = self.wr[k] - self.mu * (er * vr + ei * vi)
            self.wi[k] = self.wi[k] - self.mu * (ei * vr - er * vi)
        return yr, yi


# ---- channels as array rows ----------------------------------------------------------------------------------------------
class FseBatch(CmaBatch):
    def __init__(self, n_taps, mu, modulus=1.0, channels=1, sps=1):
        check_params(n_taps, mu, modulus, sps)
        self.sps = int(sps)
        super().__init__(n_taps, mu, modulus, channels)

    def reset(self):
        super().reset()
        self.phase = np.zeros(self.C, np.int64)      # stream sample counter mod sps

    def process(self, x, lengths=None, drop=False):
        """as CmaBatch.process; the taps of channel c update on its samples t with (phase[c] + t) % sps == 0"""
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
            upd = (act & ((self.phase + t) % self.sps == 0))[:, None]
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
            self.wr = np.where(upd, self.wr - mu * gr, self.wr)
            self.wi = np.where(upd, self.wi - mu * gi, self.wi)
            self.vr, self.vi = vr, vi
            yr_all[:, t], yi_all[:, t] = yr, yi
        self.phase = (self.phase + n) % self.sps
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


# ---- the oracle demodulator with both stages ------------------------------------------------------------------------------
class FseDemod(EqDemod):
    """EqDemod with the fractionally spaced stage between the matched filter and Mueller-Muller (set_fractional_equalizer);
    with that stage off it is EqDemod."""

    def __init__(self, orc, fs, rs, *args, **kw):
        super().__init__(orc, fs, rs, *args, **kw)
        self.fs, self.rs = fs, rs
        self.fse = None

    def set_fractional_equalizer(self, n_taps, mu, modulus=1.0):
        """update stride S = fs / rs: needs fs % rs == 0 and S in 2..8 (else status -7, before the other checks)"""
        if n_taps == 0:
            self.fse = None
            return
        sps = self.fs // self.rs if self.fs % self.rs == 0 else 0
        if not 2 <= sps <= MAX_SPS:
            raise EqArgumentError(-7)
        check_params(n_taps, mu, modulus, sps)
        self.fse = FseBatch(n_taps, mu, modulus, self.C, sps=sps)

    def fractional_equalizer_taps(self):
        return self.fse.taps

    def _symbols(self, rx):
        if self.fse is None:
            return super()._symbols(rx)
        rx = np.asarray(rx, np.float32).reshape(self.C, -1)
        mf = []
        for c in range(self.C):
            x = rx[c]
            if self.use_fll:
                x = self.fll[c].Process(x)
            mf.append(self.rrc[c].Filter(x))
        mf = self.fse.process(np.stack(mf), drop=True)          # every channel has the call's L samples
        syms = [self.mm[c].Process(m) for c, m in enumerate(mf)]
        if self.eq is None:
            return syms
        L = max(s.size for s in syms) if syms else 0
        pad = np.zeros((self.C, max(L, 2)), np.float32)
        for c, s in enumerate(syms):
            pad[c, : s.size] = s
        return self.eq.process(pad, [s.size // 2 for s in syms], drop=True)
