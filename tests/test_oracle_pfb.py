"""CPU: the fp64 restatements of the polyphase analysis channelizer (tests/pfb_oracle.py) agree with each other, the
host-side prototype designer qpsk_pfb_taps matches scipy.signal.firwin, a tone lands in its channel with the stated gain
and phase, and a 4-of-16 QPSK scene goes wideband -> channels -> payloads through the CPU oracle's demodulator.  No GPU."""
import ctypes as C

import numpy as np
import pytest
from scipy.signal import firwin, kaiser_beta

from pfb_oracle import SCENE_FS, SCENE_RS, TSC, PfbPoly, pfb_direct, qpsk_fdm_scene, scene_channels


def _cx(rng, n):
    return rng.standard_normal(n) + 1j * rng.standard_normal(n)


@pytest.mark.parametrize("M,n_taps", [(2, 1), (2, 7), (4, 16), (8, 61), (16, 128), (32, 33), (64, 500), (128, 4096)])
def test_direct_and_polyphase_agree(M, n_taps):
    rng = np.random.default_rng(M * 1000 + n_taps)
    h = rng.standard_normal(n_taps)
    x = _cx(rng, 7 * M + 5 + 3 * (n_taps // M) * M)          # ragged: not a whole number of blocks
    want = pfb_direct(h, M, x)
    got = PfbPoly(h, M).process(x)
    assert got.shape == want.shape
    assert np.abs(got - want).max() <= 1e-12 * np.abs(want).max()
    # the same stream in chunks, including 0, 1 and M-1 samples
    p = PfbPoly(h, M)
    cuts = [0, 1, M - 1, 0, M, 2 * M + 1, 3, 0]
    parts, a = [], 0
    for c in cuts:
        parts.append(p.process(x[a:a + c]))
        a += c
    parts.append(p.process(x[a:]))
    chunked = np.concatenate(parts, axis=1)
    assert np.abs(chunked - want).max() <= 1e-12 * np.abs(want).max()
    p.reset()
    assert np.abs(p.process(x) - want).max() <= 1e-12 * np.abs(want).max()


@pytest.mark.parametrize("M,P,cutoff,atten", [(2, 1, 0.25, 60.0), (16, 8, 0.5 / 16, 60.0), (64, 16, 0.4 / 64, 80.0),
                                              (1024, 32, 0.5 / 1024, 45.0), (8, 4, 0.1, 15.0), (256, 3, 0.6 / 256, 100.0)])
def test_prototype_designer_matches_firwin(qp, M, P, cutoff, atten):
    h = qp.pfb_taps(M, P, cutoff, atten)
    want = firwin(M * P, 2 * cutoff, window=("kaiser", kaiser_beta(atten)), scale=True)
    assert h.size == M * P
    assert np.abs(h - want).max() <= 1e-12 * np.abs(want).max()
    assert abs(h.sum() - 1.0) < 1e-12


def test_prototype_designer_size_query_and_limits(qp):
    L = qp._native.lib()
    n = C.c_int(0)
    assert L.qpsk_pfb_taps(16, 8, 0.03, 60.0, None, 0, C.byref(n)) == 0 and n.value == 128
    buf = (C.c_double * 127)()
    n.value = 0
    assert L.qpsk_pfb_taps(16, 8, 0.03, 60.0, buf, 127, C.byref(n)) == qp._native.ERR_CAPACITY and n.value == 128
    for args, st in [((12, 8, 0.03, 60.0), qp._native.ERR_UNSUPPORTED), ((2048, 8, 0.03, 60.0), qp._native.ERR_UNSUPPORTED),
                     ((16, 33, 0.03, 60.0), qp._native.ERR_UNSUPPORTED), ((16, 0, 0.03, 60.0), qp._native.ERR_UNSUPPORTED),
                     ((16, 8, 0.0, 60.0), qp._native.ERR_RANGE), ((16, 8, 0.5, 60.0), qp._native.ERR_RANGE),
                     ((16, 8, 0.03, float("nan")), qp._native.ERR_RANGE), ((16, 8, 0.03, -1.0), qp._native.ERR_RANGE)]:
        assert L.qpsk_pfb_taps(*args, None, 0, C.byref(n)) == st, args
    assert L.qpsk_pfb_taps(16, 8, 0.03, 60.0, None, 0, None) == qp._native.ERR_NULL


@pytest.mark.parametrize("M,k0", [(16, 3), (16, 13), (64, 0), (64, 40)])
def test_tone_lands_in_its_channel_with_unit_gain_and_the_stated_phase(qp, M, k0):
    h = qp.pfb_taps(M, 8, 0.5 / M, 60.0)
    f = (k0 + 0.1) / M
    n = 64 * M
    t = np.arange(n)
    x = np.exp(2j * np.pi * f * t)
    y = PfbPoly(h, M).process(x)[:, 8:]                         # past the P-block start-up
    m = np.arange(8, n // M)
    N = m * M + M - 1
    # mix down by k0/M, filter, keep n = N; the channelizer's output is that times e^{-j 2 pi k0 / M}
    base = np.array([np.sum(h * x[Ni - np.arange(h.size)] * np.exp(-2j * np.pi * k0 * (Ni - np.arange(h.size)) / M)) for Ni in N])
    assert np.abs(y[k0] - np.exp(-2j * np.pi * k0 / M) * base).max() < 1e-9
    assert np.abs(np.abs(y[k0]) - 1.0).max() < 2e-3                 # unit gain within the passband ripple
    # the tone's offset from the channel centre, seen through the prototype's group delay (L-1)/2, and the channel's phase
    want = np.exp(2j * np.pi * (0.1 / M) * (N - (h.size - 1) / 2)) * np.exp(-2j * np.pi * k0 / M)
    assert np.abs(np.angle(y[k0] / want)).max() < 2e-3
    p_in = np.mean(np.abs(y[k0]) ** 2)
    for k in range(M):
        if k != k0:
            assert 10 * np.log10(np.mean(np.abs(y[k]) ** 2) / p_in) <= -50.0, k


def test_qpsk_scene_through_the_cpu_channelizer_and_oracle_demodulator(qp, orc):
    M = 16
    h = qp.pfb_taps(M, 8, 0.5 / M, 60.0)
    occ = scene_channels(M, 4)
    wide, pays = qpsk_fdm_scene(orc, h, M, occ, seed=5)
    y = PfbPoly(h, M).process(wide)
    for k in range(M):
        iq = np.ascontiguousarray(y[k].astype(np.complex64)).view(np.float32)
        got = orc.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC).DeModulateBytes(iq, b"START", b"END")
        assert got == pays.get(k, b""), k
