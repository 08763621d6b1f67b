"""CPU: the restatement of the Reed-Solomon outer code (tests/rs_oracle.py).  The generator has exactly the roots
alpha^0..alpha^(nroots-1); every codeword has zero syndromes and the encoder is linear; the round trip with up to t symbol
errors anywhere (parity included, interleaved blocks included) is exact; beyond t the decoder fails or lands on a codeword
within t; brute force over every codeword of tiny shortened codes confirms the decoding rule exactly; and, behind the
Viterbi decoder of tests/fec_oracle.py, depth-4 RS(255, 223) clears every codeword at Eb/N0 = 3 dB where Viterbi alone
leaves byte errors in two thirds of them."""
import numpy as np
import pytest

import rs_oracle as R


_errors = R.add_errors


@pytest.mark.parametrize("nroots", [2, 4, 16, 32])
def test_generator_roots(nroots):
    g = R.generator(nroots)
    assert g.size == nroots + 1 and g[-1] == 1
    vals = R.poly_eval(g[::-1][None], R.gpow(np.arange(255))[:, None])[:, 0]
    assert np.array_equal(np.nonzero(vals == 0)[0], np.arange(nroots))


def test_gf_tables():
    assert R.EXP[8] == 0x1D and R.EXP[255] == 1 and len(set(R.EXP[:255].tolist())) == 255
    a = np.arange(256)
    assert np.array_equal(R.gmul(a, 1), a) and not R.gmul(a, 0).any()
    nz = a[1:]
    assert (R.gmul(nz, R.gdiv(1, nz)) == 1).all()


@pytest.mark.parametrize("nroots,k", [(2, 1), (4, 7), (16, 48), (32, 223), (32, 1), (16, 239), (4, 251)])
def test_codewords_have_zero_syndromes_and_the_encoder_is_linear(nroots, k):
    c = R.Code(nroots, k)
    rng = np.random.default_rng(nroots * 1000 + k)
    a, b = rng.integers(0, 256, (2, 20, k))
    ea, eb, ex = c.encode_words(a), c.encode_words(b), c.encode_words(a ^ b)
    assert np.array_equal(ea[:, :k], a)                                   # systematic
    assert not c.syndromes(ea).any() and not c.syndromes(eb).any()
    assert np.array_equal(ex, ea ^ eb)
    # the parity is m(x) x^nroots mod g(x): m(x) x^nroots + parity(x) is a multiple of g
    assert not R.poly_eval(ea, R.gpow(np.arange(nroots))[:, None]).any()


@pytest.mark.parametrize("depth", [1, 4, 8])
@pytest.mark.parametrize("nroots", [2, 4, 16, 32])
@pytest.mark.parametrize("kind", ["one", "small", "full"])
def test_round_trip_up_to_t_errors(nroots, kind, depth):
    k = {"one": 1, "small": 9, "full": 255 - nroots}[kind]
    c = R.Code(nroots, k, depth)
    rng = np.random.default_rng(nroots * 31 + k * 7 + depth)
    nb = 6
    msg = rng.integers(0, 256, nb * depth * k).astype(np.uint8)
    code = c.encode(msg)
    assert code.size == nb * depth * c.n
    assert np.array_equal(code.reshape(nb, -1)[:, : depth * k].ravel(), msg)  # the message stays in place
    words = c.deinterleave(code)
    counts = rng.integers(0, c.t + 1, words.shape[0])
    counts[:2] = (0, c.t)
    rx = c.interleave(_errors(rng, words, counts))
    got, st = c.decode(rx)
    assert np.array_equal(got, msg)
    assert np.array_equal(st, counts)
    # a remainder past the last whole block is ignored
    got2, st2 = c.decode(np.concatenate([rx, np.full(depth * c.n - 1, 7, np.uint8)]))
    assert np.array_equal(got2, msg) and np.array_equal(st2, st)


@pytest.mark.parametrize("nroots,k", [(4, 20), (16, 48), (32, 223)])
def test_beyond_t_fails_or_lands_within_t(nroots, k):
    c = R.Code(nroots, k)
    rng = np.random.default_rng(nroots + k)
    words = c.encode_words(rng.integers(0, 256, (400, k)))
    counts = rng.integers(c.t + 1, min(c.n, 3 * c.t + 2), 400)
    rx = _errors(rng, words, counts)
    got, st = c.decode_words(rx)
    fail = st < 0
    assert fail.any()
    assert np.array_equal(got[fail], rx[fail])
    ok = ~fail
    assert not c.syndromes(got[ok]).any()
    assert np.array_equal((got[ok] != rx[ok]).sum(axis=1), st[ok])
    assert (st[ok] <= c.t).all()


def test_rule_brute_force_t1_every_single_symbol_change():
    """RS(4, 2), t = 1: from a codeword and from a word at distance 2 of one, every single-symbol change decodes exactly
    as the nearest-codeword rule says."""
    c = R.Code(2, 2)
    rng = np.random.default_rng(7)
    cw = c.encode_words(rng.integers(0, 256, (1, 2)))[0]
    far = cw.copy()
    far[[0, 3]] ^= np.array([5, 9], np.uint8)
    for base in (cw, far):
        words = np.repeat(base[None], c.n * 255, axis=0)
        for p in range(c.n):
            words[p * 255:(p + 1) * 255, p] ^= np.arange(1, 256, dtype=np.uint8)
        got, st = c.decode_words(words)
        want, wst = R.brute_decode(c, words)
        assert np.array_equal(st, wst) and np.array_equal(got, want)
        if base is cw:
            assert (st == 1).all()
        else:
            assert (st == 1).any() and (st == -1).any()


@pytest.mark.parametrize("k", [1, 2])
def test_rule_brute_force_t2_short_code(k):
    """RS(4 + k, k), t = 2: random words at every distance from a codeword, and uniformly random words: a word decodes if
    and only if a codeword lies within t, and then to that codeword."""
    c = R.Code(4, k)
    rng = np.random.default_rng(11 + k)
    N = 1500
    words = c.encode_words(rng.integers(0, 256, (N, k)))
    rx = _errors(rng, words, rng.integers(0, c.n + 1, N))
    rx[-200:] = rng.integers(0, 256, (200, c.n))
    got, st = c.decode_words(rx)
    want, wst = R.brute_decode(c, rx)
    assert np.array_equal(st, wst) and np.array_equal(got, want)
    assert (st == -1).sum() > 50 and (st == 2).sum() > 50


def test_concatenated_gain_at_3_db():
    """Coherent AWGN at Eb/N0 = 3.0 dB per information bit, 128 channels x one depth-4 RS(255, 223) block: Viterbi alone
    leaves byte errors in 68 % of the 512 codewords (at most 7 in one, 4.6e-3 of the bytes); after RS no codeword fails
    and every message is exact."""
    code = R.Code(32, 223, 4)
    msg, sent, got = R.viterbi_chain(np.random.default_rng(300), code, 128, 3.0)
    dirty = np.concatenate([(code.deinterleave(g) != code.deinterleave(s)).any(axis=1) for g, s in zip(got, sent)])
    assert dirty.size == 512 and 0.4 < dirty.mean() < 0.9, dirty.mean()
    for m, g in zip(msg, got):
        out, st = code.decode(g)
        assert (st >= 0).all() and np.array_equal(out, m)


def test_decode_rows_reads_the_device_layout():
    c = R.Code(4, 5, 2)
    rng = np.random.default_rng(3)
    rows = np.zeros((5, 60), np.uint8)
    msgs = [rng.integers(0, 256, b * 10).astype(np.uint8) for b in (0, 1, 2, 3, 1)]
    for r, m in enumerate(msgs):
        rows[r, : m.size // 10 * 18] = c.encode(m)
    counts = np.array([17, 18 + 5, 36, 999, -4])
    out = c.decode_rows(rows, counts)
    assert [o[0].size for o in out] == [0, 10, 20, 30, 0]
    assert [o[1].size for o in out] == [0, 2, 4, 6, 0]
    assert np.array_equal(out[1][0], msgs[1]) and np.array_equal(out[2][0], msgs[2]) and np.array_equal(out[3][0], msgs[3])
