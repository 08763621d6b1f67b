"""GPU parity of every FLL kernel instantiation (tests/kernel_variants.py: FLL_ROWS) against oracle.FLLBandEdgeFilter, bit for
bit, outputs and the final (phase, freq) of every compared channel: fll_duo_kernel<K, TAIL, PAIRS> for N = 8..55 at 5 streams
(PAIRS = 1) and at 1300 streams (PAIRS = 4, 82 CTAs, the last with one live pair and three idle ones), the switch at
1280 / 1281 streams, fll_pair_kernel at 5120 streams, and the generic fll_group_kernel from 1 to 1430 taps (from 287 taps on
its shared memory needs the opt-in above 48 KiB).  Channel c carries input stream c mod 37 and starts from its own loop
state, so a channel that read another's samples, ring or state would differ from its oracle."""
import ctypes as C_
import os

import numpy as np
import pytest

import kernel_variants as kv

pytestmark = pytest.mark.gpu

U32 = np.uint32
STREAMS = 37
SPS, ROLLOFF, BW = 4.0, 0.35, 0.05
# call lengths in complex samples: shorter than one 4-sample hand-over batch, shorter than every two-warp N, odd lengths
CUTS = (3, 7, 1, 61, 200, 333, 95)
L = sum(CUTS)


def _inputs(orc):
    """37 streams of noise under a carrier offset of their own, so the loop moves, wraps and clamps differently in each."""
    n = np.arange(L)
    out = np.empty((STREAMS, 2 * L), np.float32)
    for s in range(STREAMS):
        z = orc.fill_uniform(11, s, 0, 2 * L).astype(np.float64)
        z = (z[0::2] + 1j * z[1::2]) * np.exp(2j * np.pi * (0.004 * (s % 9 - 4)) * n + 1j * s)
        out[s, 0::2], out[s, 1::2] = z.real, z.imag
    return out


def _start_state(C):
    c = np.arange(C)
    phase = (((c * 7.3) % 62.0) - 31.0).astype(np.float32)            # |phase| < 32: no far-phase detour
    freq = (0.002 * ((c % 7) - 3)).astype(np.float32)
    return phase, freq


def _compared(C):
    if C <= 64:
        return list(range(C))
    last_cta = (C - 1) // 16 * 16
    picks = {0, C - 1, 3, 4, 15, 16, last_cta - 1} | set(range(last_cta, C)) | set(range(0, C, STREAMS))
    return sorted(picks)


@pytest.fixture(scope="module")
def streams(orc):
    return _inputs(orc)


@pytest.mark.parametrize("n_taps,channels", kv.FLL_ROWS)
def test_fll_variant_matches_oracle(gpu, orc, streams, n_taps, channels):
    X = streams[np.arange(channels) % STREAMS]
    ph, fr = _start_state(channels)
    g = gpu.FLLBandEdgeFilter(SPS, ROLLOFF, n_taps, BW, channels=channels)
    g.state = (ph, fr)
    outs, a = [], 0
    for n in CUTS:
        part = np.ascontiguousarray(X[:, 2 * a: 2 * (a + n)])
        outs.append(g.Process(part if channels > 1 else part[0]).reshape(channels, -1))
        a += n
    got = np.concatenate(outs, axis=1)
    gp, gf = (np.atleast_1d(np.asarray(v, np.float32)) for v in g.state)
    for c in _compared(channels):
        o = orc.FLLBandEdgeFilter(SPS, ROLLOFF, n_taps, BW)
        o.state = (float(ph[c]), float(fr[c]))
        want, a = [], 0
        for n in CUTS:
            want.append(o.Process(X[c, 2 * a: 2 * (a + n)]))
            a += n
        want = np.concatenate(want)
        assert np.array_equal(got[c].view(U32), want.view(U32)), (n_taps, channels, c, int(np.argmax(got[c] != want)))
        op, of = o.state
        assert (np.float32(op), np.float32(of)) == (gp[c], gf[c]), (n_taps, channels, c)


def test_fll_launches_the_predicted_kernels(gpu):
    got = kv.launched_in_child("fll", int(os.environ.get("LOCAL_RANK", "0")))
    assert got == kv.predicted_launches("fll")


def test_fll_create_limit_on_the_device(gpu):
    """1430 taps creates and runs; 1431 is refused by the FLL and by the chain that embeds one."""
    lib, N = gpu._native.lib(), gpu._native
    h = C_.c_void_p()
    assert lib.qpsk_fll_create(SPS, ROLLOFF, 1431, BW, C_.byref(h)) == N.ERR_UNSUPPORTED
    g = gpu.FLLBandEdgeFilter(SPS, ROLLOFF, 1430, BW)
    assert g.Process(np.ones(64, np.float32)).shape == (64,)
    p = N.ChainParams()
    assert lib.qpsk_chain_default_params(C_.byref(p)) == 0
    p.fll_size = 1431
    assert lib.qpsk_chain_create(C_.byref(p), 2, C_.byref(h)) == N.ERR_UNSUPPORTED
    p.fll_size = 1430
    assert lib.qpsk_chain_create(C_.byref(p), 2, C_.byref(h)) == 0
    lib.qpsk_chain_destroy(h)
