"""CPU restatement of the convolutional code and the Viterbi decoder of csrc/fec.cu (definition in include/qpskcuda.h).

Written from the definition, not from the kernel: the GPU must be bit-identical to it.
  * code: K = 7, rate 1/2, generators 171 and 133 (octal); register s = (u << 6) | S, S the last six inputs (newest at
    bit 5); pair (parity(s & 0o171), parity(s & 0o133)), c0 first; next state s >> 1.
  * soft values: q(v) = clamp(rint_half_even(v), -127, 127), NaN -> 0, every operation a separately rounded fp32 one
    (numpy float32 arithmetic rounds each operation; nothing is fused).
  * add-compare-select: branch metric sum_i (c_i ? -s_i : s_i); predecessors of S' are 2j, 2j+1 (j = S' & 31), a tie keeps
    2j; metrics start at 0.  Metrics are int64 here and never renormalised: comparisons are exact either way.
  * decisions: B = 32, D = 64; after absolute step (k+1)B + D - 1 the bits of steps [kB, (k+1)B) are read off the survivor
    of the best state (minimum metric, lowest state on ties); flush reads the rest off the best state at the last step.
Everything is vectorised over channels; every decision of a stream is kept (one uint64 per step)."""
import numpy as np

B, D = 32, 64
G0, G1 = 0o171, 0o133
DEFAULT_SCALE = {False: 32.0, True: 24.0}        # QPSK_VITERBI_SCALE_COHERENT / _DIFFERENTIAL


def parity(x):
    x = np.asarray(x, np.int64)
    p = np.zeros_like(x)
    for k in range(7):
        p ^= (x >> k) & 1
    return p


# per new state S' (64) and predecessor choice b (2): the register and its code pair
_SP = np.arange(64)
_PRED = np.stack([((_SP & 31) << 1), ((_SP & 31) << 1) | 1], axis=1)            # [64, 2]
_REG = ((_SP >> 5) << 6)[:, None] | _PRED                                        # [64, 2]
_C0, _C1 = parity(_REG & G0), parity(_REG & G1)


def encode(bits, state=None):
    """bits [C, n] 0/1 -> ([C, 2n] 0/1, final state [C]).  `state` carries the six-bit register across calls."""
    bits = np.atleast_2d(np.asarray(bits, np.uint8)) != 0
    Cn, n = bits.shape
    S = np.zeros(Cn, np.int64) if state is None else np.asarray(state, np.int64).copy()
    out = np.zeros((Cn, 2 * n), np.uint8)
    for k in range(n):
        s = (bits[:, k].astype(np.int64) << 6) | S
        out[:, 2 * k] = parity(s & G0)
        out[:, 2 * k + 1] = parity(s & G1)
        S = s >> 1
    return out, S


def q(v):
    v = np.asarray(v, np.float32)
    with np.errstate(invalid="ignore"):
        r = np.where(np.isnan(v), np.float32(0), np.clip(np.rint(v), -127, 127))
        return r.astype(np.int64)


def soft_coherent(y, scale):
    y = np.asarray(y, np.complex64)
    sc = np.float32(scale)
    with np.errstate(over="ignore", invalid="ignore"):      # inf and NaN are part of the definition
        return q(sc * y.real.astype(np.float32)), q(sc * y.imag.astype(np.float32))


def soft_differential(y, p, scale):
    """z = y conj(p) with re = yr*pr + yi*pi, im = yi*pr - yr*pi; s0 = q(-(scale*(re+im))), s1 = q(scale*(im-re))."""
    yr, yi = np.float32(y.real), np.float32(y.imag)
    pr, pi = np.float32(p.real), np.float32(p.imag)
    yr, yi, pr, pi = (np.asarray(a, np.float32) for a in (yr, yi, pr, pi))
    sc = np.float32(scale)
    with np.errstate(over="ignore", invalid="ignore"):
        re = yr * pr + yi * pi
        im = yi * pr - yr * pi
        return q(-(sc * (re + im))), q(sc * (im - re))


def branch_metrics(s0, s1):
    """s0, s1 [C] -> [C, 64, 2]: metric of the branch from predecessor b of each new state."""
    s0, s1 = np.asarray(s0, np.int64)[:, None, None], np.asarray(s1, np.int64)[:, None, None]
    return np.where(_C0, -s0, s0) + np.where(_C1, -s1, s1)


def emitted(n):
    """steps emitted after n steps"""
    n = np.asarray(n, np.int64)
    return np.where(n >= D, ((n - D) // B) * B, 0)


class Viterbi:
    """Streaming decoder over `channels`; decode / flush take complex64 rows and per-channel counts."""

    def __init__(self, channels=1, differential=True, scale=None):
        self.C, self.diff = channels, bool(differential)
        self.scale = np.float32(DEFAULT_SCALE[self.diff] if scale is None else scale)
        self.reset()

    def reset(self):
        self.M = np.zeros((self.C, 64), np.int64)
        self.n = np.zeros(self.C, np.int64)                   # steps processed
        self.dec = np.zeros((self.C, 256), np.uint64)         # decisions of step t at [c, t]: bit S for new state S
        self.prev = np.zeros(self.C, np.complex64)
        self.have = np.zeros(self.C, bool)

    def _steps(self, s0, s1, act):
        """one trellis step for the channels in `act` (bool [C]), soft values s0, s1 [C]"""
        bm = branch_metrics(s0, s1)
        cand = self.M[:, _PRED] + bm                          # [C, 64, 2]
        d = cand[:, :, 1] < cand[:, :, 0]
        newM = np.where(d, cand[:, :, 1], cand[:, :, 0])
        self.M = np.where(act[:, None], newM, self.M)
        words = (d.astype(np.uint64) << np.arange(64, dtype=np.uint64)).sum(axis=1, dtype=np.uint64)
        if int(self.n.max()) >= self.dec.shape[1]:
            self.dec = np.concatenate([self.dec, np.zeros_like(self.dec)], axis=1)
        idx = np.nonzero(act)[0]
        self.dec[idx, self.n[idx]] = words[idx]
        self.n += act

    def _trace(self, cs, stop):
        """channels cs: bits of steps [stop[c], n[c]) off the survivor of the best state at step n[c] - 1, as a list"""
        n = self.n[cs]
        S = np.argmin(self.M[cs], axis=1).astype(np.int64)    # argmin returns the lowest state on ties
        L = n - stop
        out = np.zeros((cs.size, int(L.max()) if cs.size else 0), np.uint8)
        for a in range(out.shape[1]):                         # a steps back from the last
            t = n - 1 - a
            live = a < L
            out[live, (t - stop)[live]] = (S[live] >> 5).astype(np.uint8)
            w = self.dec[cs, np.maximum(t, 0)]
            b = ((w >> S.astype(np.uint64)) & np.uint64(1)).astype(np.int64)
            S = np.where(live, ((S & 31) << 1) | b, S)
        return [out[k, : L[k]] for k in range(cs.size)]

    def _run(self, sym, n_sym, flush):
        sym = np.asarray(sym, np.complex64).reshape(self.C, -1)
        n_sym = np.broadcast_to(np.asarray(n_sym, np.int64), (self.C,)).copy()
        out = [[] for _ in range(self.C)]
        first = np.zeros(self.C, np.int64)
        if self.diff and sym.shape[1]:                        # the first symbol ever seen yields no step
            take = ~self.have & (n_sym > 0)
            self.prev = np.where(take, sym[:, 0], self.prev)
            self.have |= take
            first = take.astype(np.int64)
        for i in range(int(n_sym.max()) if self.C else 0):
            act = (i >= first) & (i < n_sym)
            if not act.any():
                continue
            y = sym[:, i]
            if self.diff:
                s0, s1 = soft_differential(y, self.prev, self.scale)
                self.prev = np.where(act, y, self.prev)
            else:
                s0, s1 = soft_coherent(y, self.scale)
            self._steps(s0, s1, act)
            due = np.nonzero(act & (self.n % B == 0) & (self.n >= B + D))[0]
            if due.size:
                for c, bits in zip(due, self._trace(due, self.n[due] - B - D)):
                    out[c].append(bits[:B])
        if flush:
            cs = np.arange(self.C)
            for c, bits in zip(cs, self._trace(cs, emitted(self.n))):
                out[c].append(bits)
        res = [np.concatenate(o).astype(np.uint8) if o else np.zeros(0, np.uint8) for o in out]
        if flush:
            self.reset()
        return res

    def decode(self, sym, n_sym):
        return self._run(sym, n_sym, False)

    def flush(self, sym=None, n_sym=0):
        if sym is None:
            sym = np.zeros((self.C, 0), np.complex64)
        return self._run(sym, n_sym, True)


def path_metric(soft0, soft1, state0, inputs):
    """metric of the path that starts in `state0` and takes `inputs` (one channel, soft values per step)"""
    S, m = int(state0), 0
    for k, u in enumerate(inputs):
        s = (int(u) << 6) | S
        c0, c1 = int(parity(s & G0)), int(parity(s & G1))
        m += (-soft0[k] if c0 else soft0[k]) + (-soft1[k] if c1 else soft1[k])
        S = s >> 1
    return m


def qpsk_symbols(coded, differential, rng_phase=0):
    """coded bits [C, 2n] -> unit-amplitude symbols [C, n (+1 with a reference symbol when differential)].
    Coherent: I = c0 ? +1 : -1, Q = c1 ? +1 : -1, over sqrt 2.  Differential: delta 00 -> +1, 01 -> +j, 11 -> -1, 10 -> -j
    applied to a running symbol that starts at (1 + j)/sqrt 2 (the first symbol is the reference)."""
    coded = np.atleast_2d(np.asarray(coded, np.int64))
    c0, c1 = coded[:, 0::2], coded[:, 1::2]
    if not differential:
        return ((2 * c0 - 1) + 1j * (2 * c1 - 1)).astype(np.complex64) / np.float32(np.sqrt(2))
    quad = np.select([(c0 == 0) & (c1 == 0), (c0 == 0) & (c1 == 1), (c0 == 1) & (c1 == 1)], [0, 1, 2], 3)
    acc = np.concatenate([np.zeros((coded.shape[0], 1), np.int64), np.cumsum(quad, axis=1)], axis=1) + rng_phase
    return (np.exp(1j * (np.pi / 4 + np.pi / 2 * acc))).astype(np.complex64)
