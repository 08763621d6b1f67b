"""CPU: the restatement of the convolutional code and the Viterbi decoder (tests/fec_oracle.py).  The encoder's impulse
response and linearity; the decoder is maximum-likelihood (brute force over every start state and input sequence for up
to 12 steps); the noiseless round trip is exact in both modes; coding gain on a coherent AWGN channel at Eb/N0 = 4.5 dB;
any split of the symbols over calls gives the same bits; the differential soft values carry the hard decisions of the
reference's map."""
import itertools

import numpy as np
import pytest

import fec_oracle as F


def test_impulse_response_and_linearity():
    out, S = F.encode(np.array([[1, 0, 0, 0, 0, 0, 0]]))
    assert "".join(map(str, out[0])) == "11101111000111"            # 11 10 11 11 00 01 11
    assert S[0] == 0
    rng = np.random.default_rng(0)
    a, b = rng.integers(0, 2, (2, 4, 300))
    ea, eb, ex = F.encode(a)[0], F.encode(b)[0], F.encode(a ^ b)[0]
    assert np.array_equal(ex, ea ^ eb)


def test_encoder_state_carries_across_calls():
    rng = np.random.default_rng(1)
    bits = rng.integers(0, 2, (3, 257))
    whole = F.encode(bits)[0]
    st, parts = None, []
    for lo, hi in ((0, 0), (0, 1), (1, 64), (64, 64), (64, 257)):
        o, st = F.encode(bits[:, lo:hi], st)
        parts.append(o)
    assert np.array_equal(np.concatenate(parts, axis=1), whole)


def _brute_min(s0, s1):
    """minimum path metric over every start state and input sequence of len(s0) steps (vectorised over sequences)"""
    n = len(s0)
    u = np.array(list(itertools.product((0, 1), repeat=n)), np.int64)      # [2^n, n]
    best = None
    for st in range(64):
        S = np.full(u.shape[0], st, np.int64)
        m = np.zeros(u.shape[0], np.int64)
        for k in range(n):
            s = (u[:, k] << 6) | S
            c0, c1 = F.parity(s & F.G0), F.parity(s & F.G1)
            m += np.where(c0 == 1, -s0[k], s0[k]) + np.where(c1 == 1, -s1[k], s1[k])
            S = s >> 1
        v = int(m.min())
        best = v if best is None else min(best, v)
    return best


@pytest.mark.parametrize("n", [1, 2, 5, 6, 7, 9, 12])
def test_decoder_is_maximum_likelihood(n):
    rng = np.random.default_rng(100 + n)
    for trial in range(3):
        s0 = rng.integers(-127, 128, n)
        s1 = rng.integers(-127, 128, n)
        if trial == 2:                                   # many ties
            s0, s1 = rng.integers(-2, 3, n), rng.integers(-2, 3, n)
        sym = (s0 + 1j * s1).astype(np.complex64)[None]
        got = F.Viterbi(1, False, scale=1.0).flush(sym, n)[0]
        assert got.size == n
        decoded = min(F.path_metric(s0, s1, st, got) for st in range(64))
        assert decoded == _brute_min(s0, s1), (n, trial)


@pytest.mark.parametrize("differential", [False, True])
def test_noiseless_round_trip(differential):
    rng = np.random.default_rng(2)
    bits = rng.integers(0, 2, (6, 700)).astype(np.uint8)
    y = F.qpsk_symbols(F.encode(bits)[0], differential)
    got = F.Viterbi(6, differential).flush(y, y.shape[1])
    for g, b in zip(got, bits):
        assert np.array_equal(g, b)


def test_coding_gain_at_4_5_db():
    """Coherent AWGN, Eb/N0 = 4.5 dB per information bit, 2^18 information bits: decoded BER < 1e-4, where uncoded hard
    decisions at the same Eb/N0 lose about 9e-3."""
    ebn0 = 10 ** (4.5 / 10)
    rng = np.random.default_rng(45)
    Cn, n = 64, 4096
    bits = rng.integers(0, 2, (Cn, n)).astype(np.uint8)
    y = F.qpsk_symbols(F.encode(bits)[0], False)
    sig = np.sqrt(0.5 / ebn0)                             # one information bit per unit-energy symbol
    y = (y + sig * (rng.standard_normal(y.shape) + 1j * rng.standard_normal(y.shape))).astype(np.complex64)
    got = F.Viterbi(Cn, False).flush(y, y.shape[1])
    errs = sum(int((g != b).sum()) for g, b in zip(got, bits))
    assert errs / bits.size < 1e-4, errs
    # uncoded QPSK at the same Eb/N0 carries two information bits per symbol
    sig_u = np.sqrt(0.25 / ebn0)
    ref = rng.integers(0, 2, 1 << 18)
    hard = ((2 * ref - 1) / np.sqrt(2) + sig_u * rng.standard_normal(ref.size)) > 0
    assert 7e-3 < np.mean(hard != ref) < 1.1e-2


def _split(rng, n):
    cuts, a = [], 0
    while a < n:
        c = int(rng.choice([0, 1, 2, 31, 32, 33, int(rng.integers(0, 100))]))
        cuts.append(min(c, n - a))
        a += cuts[-1]
    return cuts


@pytest.mark.parametrize("differential", [False, True])
def test_chunk_invariance(differential):
    rng = np.random.default_rng(3 + differential)
    Cn, n = 5, 400
    y = (rng.standard_normal((Cn, n)) + 1j * rng.standard_normal((Cn, n))).astype(np.complex64) * np.float32(0.8)
    counts = np.array([0, 1, 95, 96, 400])
    v = F.Viterbi(Cn, differential)
    whole = [np.concatenate([a, b]) for a, b in zip(v.decode(y, counts), v.flush())]
    assert [w.size for w in whole] == [max(c - differential, 0) for c in counts]
    for _ in range(2):
        v = F.Viterbi(Cn, differential)
        outs = [[] for _ in range(Cn)]
        done = np.zeros(Cn, np.int64)
        for c in _split(rng, n):
            take = np.clip(counts - done, 0, c)
            seg = np.zeros((Cn, c), np.complex64)
            for k in range(Cn):
                seg[k, : take[k]] = y[k, done[k]: done[k] + take[k]]
            for k, o in enumerate(v.decode(seg, take)):
                outs[k].append(o)
            done += take
        for k, o in enumerate(v.flush()):
            outs[k].append(o)
        for k in range(Cn):
            assert np.array_equal(np.concatenate(outs[k]), whole[k]), k


def test_decisions_are_blocked_and_delayed():
    """A decode call emits whole blocks of 32: after n steps, 32 * floor((n - 64) / 32) bits for n >= 64."""
    v = F.Viterbi(1, False)
    y = np.ones((1, 200), np.complex64)
    got = [v.decode(y[:, :k], k)[0].size for k in (95, 1, 31, 1, 72)]
    assert got == [0, 32, 0, 32, 64]
    assert v.flush()[0].size == 200 - 128                 # the 72 steps not yet emitted


def test_differential_soft_signs_match_hard_decisions():
    """Well away from the decision boundaries, the signs of the differential soft pair are the reference's dibit of
    z = y_k conj(y_{k-1}): 00 -> +1, 01 -> +j, 11 -> -1, 10 -> -j."""
    rng = np.random.default_rng(4)
    p = np.exp(1j * rng.uniform(0, 2 * np.pi, 4000)).astype(np.complex64)
    delta = rng.integers(0, 4, 4000)
    jitter = rng.uniform(-0.6, 0.6, 4000)                 # < pi/4 from the constellation point
    y = (p * np.exp(1j * (np.pi / 2 * delta + jitter))).astype(np.complex64)
    s0, s1 = F.soft_differential(y, p, 24.0)
    dibit = {0: (0, 0), 1: (0, 1), 2: (1, 1), 3: (1, 0)}
    want = np.array([dibit[d] for d in delta])
    assert np.array_equal((s0 > 0).astype(int), want[:, 0])
    assert np.array_equal((s1 > 0).astype(int), want[:, 1])


def test_soft_quantiser():
    v = np.array([0.5, 1.5, 2.5, -0.5, -1.5, 126.5, 127.5, 1e30, -1e30, np.inf, -np.inf, np.nan], np.float32)
    assert F.q(v).tolist() == [0, 2, 2, 0, -2, 126, 127, 127, -127, 127, -127, 0]
