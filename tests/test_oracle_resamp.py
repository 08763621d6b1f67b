"""CPU: the rational resampler's restatements (tests/resamp_oracle.py) agree with each other and with scipy's upfirdn, are
chunk-invariant, count outputs as the header states, pass a tone with the gain of its branch, and mirror the C limits."""
import numpy as np
import pytest
from scipy.signal import firwin, upfirdn

from resamp_oracle import (ERR_ARG, ERR_UNSUPPORTED, OK, ResampPoly, branch_taps, check_params, resamp_count,
                           resamp_direct)

RATIOS = [(1, 1), (1, 4), (4, 1), (5, 8), (8, 5), (125, 128), (1024, 1023), (3, 1024)]


def _cx(rng, *shape):
    return rng.standard_normal(shape) + 1j * rng.standard_normal(shape)


# per ratio: N < L (where L > 1), N not a multiple of L, and a full branch count
def _taps_cases(L):
    cases = [3 * L + 1, 7 * L - 1 if L > 1 else 7]
    if L > 1:
        cases.append(max(1, L // 2))
    return cases


@pytest.mark.parametrize("L,M", RATIOS)
def test_direct_poly_and_upfirdn_agree(L, M):
    rng = np.random.default_rng(L * 1031 + M)
    for N in _taps_cases(L):
        h = rng.standard_normal(N)
        n_in = max(40, 3 * M // L + 40)
        x = _cx(rng, n_in)
        n_out = resamp_count(n_in, L, M)
        # zeros past the input change no complete output, and make upfirdn's (shorter when N < L) output reach n_out
        want = upfirdn(h, np.concatenate([x, np.zeros(branch_taps(N, L) + 2)]), L, M)[:n_out]
        assert want.size == n_out
        d = resamp_direct(h, L, M, x)
        p = ResampPoly(h, L, M).process(x)[0]
        assert np.allclose(d, want, rtol=0, atol=1e-12 * np.abs(want).max())
        assert np.allclose(p, want, rtol=0, atol=1e-12 * np.abs(want).max())


def test_longest_prototype():
    rng = np.random.default_rng(1)
    L, M, N = 256, 255, 16384
    assert branch_taps(N, L) == 64
    h = rng.standard_normal(N)
    x = _cx(rng, 300)
    want = upfirdn(h, x, L, M)[:resamp_count(x.size, L, M)]
    got = ResampPoly(h, L, M).process(x)[0]
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


def test_count_formula():
    for L, M in RATIOS:
        for n in list(range(0, 50)) + [2 ** 40 + 3, 2 ** 62 - 1]:
            c = resamp_count(n, L, M)
            if n < 50:
                brute = sum(1 for m in range(n * L // M + 2) if (m * M) // L <= n - 1) if n else 0
                assert c == brute, (L, M, n)
            # the count splits as the C code computes it without overflow: (n / M) * L + count(n mod M)
            assert c == (n // M) * L + resamp_count(n % M, L, M)


@pytest.mark.parametrize("L,M", RATIOS)
def test_any_chunking_gives_identical_outputs(L, M):
    rng = np.random.default_rng(7 * L + M)
    C, N = 3, 5 * L + 2
    h = rng.standard_normal(N)
    x = _cx(rng, C, 40 * max(1, M // L) + 123)
    ref = ResampPoly(h, L, M, C).process(x)
    r = ResampPoly(h, L, M, C)
    outs, a = [], 0
    while a < x.shape[1]:
        c = min(int(rng.choice([0, 1, 1, 2, max(M // L - 1, 0), int(rng.integers(0, 60))])), x.shape[1] - a)
        before = r.n_outc
        assert r.outputs_for(c) == resamp_count(a + c, L, M) - resamp_count(a, L, M)
        outs.append(r.process(x[:, a:a + c]))
        assert r.n_outc - before == outs[-1].shape[1]
        a += c
    got = np.concatenate(outs, axis=1)
    assert got.shape == ref.shape
    assert np.array_equal(got, ref)
    r.reset()
    assert np.array_equal(r.process(x), ref)


@pytest.mark.parametrize("L,M", [(5, 8), (8, 5), (4, 1), (125, 128)])
def test_tone_gain_is_the_branch_sum(L, M):
    P = 12
    h = L * firwin(P * L, 0.8 / max(L, M), scale=True)
    hT = ResampPoly(h, L, M).hT
    # a constant input: output m equals sum_q h[phi_m + qL], the gain of its branch (once the history is full)
    x = np.ones(200 * max(1, M // L) + 3 * P, complex)
    r = ResampPoly(h, L, M)
    y = r.process(x)[0]
    m = np.arange(y.size)
    phi = (m * M) % L
    n_m = (m * M) // L
    ok = n_m >= P - 1
    assert np.allclose(y[ok].real, hT.sum(axis=1)[phi[ok]], rtol=0, atol=1e-12)
    # L * firwin(scale=True): every branch passes DC at about unit gain
    assert np.abs(hT.sum(axis=1) - 1.0).max() < 2e-3
    # and a slow tone comes out at unit amplitude
    f = 0.01 / max(1, M / L)
    xt = np.exp(2j * np.pi * f * np.arange(x.size))
    yt = ResampPoly(h, L, M).process(xt)[0][ok]
    assert np.abs(np.abs(yt) - 1.0).max() < 5e-3


def test_parameter_checks_mirror_the_c_limits():
    assert check_params(1, 1, 1, 1) == OK
    assert check_params(16384, 256, 1024, 16384) == OK
    assert check_params(64, 1, 1, 1) == OK and check_params(65, 1, 1, 1) == ERR_UNSUPPORTED      # P <= 64
    assert check_params(64 * 1024, 1024, 1, 1) == ERR_UNSUPPORTED                                # N > 16384
    assert check_params(16385, 1024, 1, 1) == ERR_UNSUPPORTED
    assert check_params(0, 1, 1, 1) == ERR_ARG and check_params(-5, 1, 1, 1) == ERR_ARG
    for L, M, C in ((0, 1, 1), (1025, 1, 1), (1, 0, 1), (1, 1025, 1), (1, 1, 0), (1, 1, 16385)):
        assert check_params(4, L, M, C) == ERR_UNSUPPORTED, (L, M, C)
