"""CPU: the fp64 restatements of the digital down-converter bank (tests/ddc_oracle.py) agree with each other under any
chunking, equal the PFB channelizer's rows times e^{+j 2 pi k / M} on a full grid, put a tone at f_k on DC of channel k
with gain sum h and zero phase, and carry an off-grid QPSK scene through the CPU oracle's demodulator.  No GPU."""
import numpy as np
import pytest

from ddc_oracle import (SCENE_D, SCENE_FREQS, SCENE_FS, SCENE_RS, TSC, DdcPoly, ddc_direct, ddc_scene, phase_angle,
                        phase_word, scene_taps)
from pfb_oracle import pfb_direct


def _cx(rng, n):
    return rng.standard_normal(n) + 1j * rng.standard_normal(n)


def test_phase_word():
    assert phase_word(0.0) == 0
    assert phase_word(0.25) == 1 << 62
    assert phase_word(-0.5) == 1 << 63
    assert phase_word(-0.25) == 3 << 62
    assert phase_word(0.5 - 2 ** -53) == (1 << 63) - (1 << 11)
    assert phase_word(2.0 ** -70) == 0 and phase_word(1.5 * 2.0 ** -64) == 2      # round half to even


@pytest.mark.parametrize("K,D,N", [(1, 1, 1), (3, 1, 17), (2, 5, 3), (4, 16, 128), (5, 7, 40), (3, 64, 100), (2, 3, 300)])
def test_direct_and_streaming_agree_under_chunking(K, D, N):
    rng = np.random.default_rng(K * 1000 + D * 10 + N)
    h = rng.standard_normal(N)
    freqs = list(rng.uniform(-0.5, 0.5, K))
    x = _cx(rng, 9 * D + N + 5)
    want = ddc_direct(h, freqs, D, x)
    got = DdcPoly(h, freqs, D).process(x)
    assert got.shape == want.shape
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    p = DdcPoly(h, freqs, D)
    parts, a = [], 0
    while a < x.size:
        c = min(int(rng.choice([0, 1, D - 1, D + 1, 2 * D + 3, int(rng.integers(0, 4 * D + 2))])), x.size - a)
        parts.append(p.process(x[a:a + c]))
        a += c
    chunked = np.concatenate(parts, axis=1)
    assert np.abs(chunked - want).max() <= 1e-12 * np.abs(want).max()
    p.reset()
    assert np.abs(p.process(x) - want).max() <= 1e-12 * np.abs(want).max()


def test_start_counter_continues_the_stream():
    """A bank started at counter S with a zero history gives what a bank fed S zeros gives next."""
    rng = np.random.default_rng(4)
    h, freqs, D = rng.standard_normal(50), [0.1234567, -0.377], 8
    S = 6 * D + 3
    x = _cx(rng, 40 * D)
    full = DdcPoly(h, freqs, D).process(np.concatenate([np.zeros(S), x]))
    got = DdcPoly(h, freqs, D, start=S).process(x)
    assert np.abs(got - full[:, S // D:]).max() <= 1e-12 * np.abs(full).max()


@pytest.mark.parametrize("M,n_taps", [(4, 16), (16, 128), (64, 300)])
def test_full_grid_equals_the_pfb_rows_times_the_channel_phase(M, n_taps):
    rng = np.random.default_rng(M + n_taps)
    h = rng.standard_normal(n_taps)
    x = _cx(rng, 20 * M + 7)
    freqs = [(k if k < M // 2 else k - M) / M for k in range(M)]
    got = DdcPoly(h, freqs, M).process(x)
    want = pfb_direct(h, M, x) * np.exp(2j * np.pi * np.arange(M) / M)[:, None]
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("D,N", [(16, 128), (5, 33), (1, 9)])
def test_tone_at_f_k_lands_on_dc_with_gain_sum_h_and_zero_phase(D, N):
    rng = np.random.default_rng(D * N)
    h = rng.standard_normal(N)
    freqs = [0.1371, -0.42, 0.0003, 0.3]
    n = 30 * D + N
    for k, f in enumerate(freqs):
        with np.errstate(over="ignore"):
            x = np.exp(1j * phase_angle(phase_word(f), np.arange(n)))
        y = DdcPoly(h, freqs, D).process(x)
        m0 = -(-(N - 1 - (D - 1)) // D) if N > D else 0             # first output whose window lies in the stream
        assert np.abs(y[k, m0:] - h.sum()).max() < 1e-12 * np.abs(h).sum()


def test_off_grid_scene_through_the_cpu_bank_and_oracle_demodulator(orc):
    h = scene_taps()
    wide, pays = ddc_scene(orc, h, SCENE_D, SCENE_FREQS, seed=5)
    y = DdcPoly(h, SCENE_FREQS, SCENE_D).process(wide)
    for k in range(len(SCENE_FREQS)):
        iq = np.ascontiguousarray(y[k].astype(np.complex64)).view(np.float32)
        got = orc.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC).DeModulateBytes(iq, b"START", b"END")
        assert got == pays[k], k
