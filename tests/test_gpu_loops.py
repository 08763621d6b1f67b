"""GPU parity: the serial loops (FLL, Mueller-Muller, Costas) one thread per stream vs the oracle.

Tolerances: loop *outputs* max |err| <= 1e-5 * max|y| (north_star).  The kernels restate the
reference arithmetic operation by operation (no FMA), and sin/cos are evaluated in fp64 and rounded
once like glibc's sinf/cosf, so in practice the outputs are bit-identical; the tests report that
and only *require* the stated tolerance.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REL_TOL = 1e-5


def _qpsk_burst(orc, nbits=2000, sps=4, span=10, alpha=0.35, seed=1, cfo=0.0, noise=0.0):
    rng = np.random.default_rng(seed)
    bits = "".join(rng.choice(["0", "1"], nbits))
    mod = orc.QPSKModulator(sps * 1000, 1000, alpha, span)
    s = mod.Modulate(bits)
    z = s[0::2] + 1j * s[1::2]
    n = np.arange(z.size)
    z = z * np.exp(1j * (2 * np.pi * cfo * n + 0.3))
    if noise > 0:
        z = z + noise * (rng.standard_normal(z.size) + 1j * rng.standard_normal(z.size))
    out = np.empty(2 * z.size, np.float32)
    out[0::2] = z.real
    out[1::2] = z.imag
    return out, bits


def _close(got, want, tol=REL_TOL):
    assert got.shape == want.shape
    if want.size == 0:
        return True
    return np.abs(got - want).max() <= tol * max(np.abs(want).max(), 1e-30)


@pytest.mark.parametrize("sps,rolloff,size,bw", [(2.0, 0.4, 40, 1e-4), (4.0, 0.35, 40, 0.01), (30.0, 0.9, 10, 0.1), (4.0, 0.5, 13, 0.05), (8.0, 1.0, 7, 0.02)])
def test_fll_matches_oracle(gpu, orc, sps, rolloff, size, bw):
    x, _ = _qpsk_burst(orc, 1500, sps=int(sps), alpha=rolloff, cfo=0.01, noise=0.02, seed=int(sps) + size)
    want_f = orc.FLLBandEdgeFilter(sps, rolloff, size, bw)
    got_f = gpu.FLLBandEdgeFilter(sps, rolloff, size, bw)
    lo_w, up_w = want_f.taps()
    lo_g, up_g = got_f.taps()
    assert np.array_equal(lo_w, lo_g) and np.array_equal(up_w, up_g)   # design is host-side fp32: exact
    cuts = [0, 2 * 700, x.size]
    for a, b in zip(cuts[:-1], cuts[1:]):                              # chunked: state carried
        want = want_f.Process(x[a:b])
        got = got_f.Process(x[a:b])
        assert _close(got, want)
    pw, fw = want_f.state
    pg, fg = got_f.state
    assert abs(pw - pg) <= 1e-4 * max(1.0, abs(pw)) and abs(fw - fg) <= 1e-5 * max(abs(fw), 1e-3)


def test_fll_batch_and_state(gpu, orc):
    C = 5
    xs = [_qpsk_burst(orc, 600, sps=4, cfo=0.002 * c, noise=0.01, seed=40 + c)[0] for c in range(C)]
    L = min(x.size for x in xs)
    x = np.stack([x[:L] for x in xs])
    f = gpu.FLLBandEdgeFilter(4.0, 0.35, 40, 0.02, channels=C)
    got = f.Process(x)
    for c in range(C):
        want = orc.FLLBandEdgeFilter(4.0, 0.35, 40, 0.02).Process(x[c])
        assert _close(got[c], want)
    g1 = gpu.FLLBandEdgeFilter(4.0, 0.35, 40, 0.02)
    g1.state = (0.5, 0.01)
    o1 = orc.FLLBandEdgeFilter(4.0, 0.35, 40, 0.02)
    o1.state = (0.5, 0.01)
    assert _close(g1.Process(x[0]), o1.Process(x[0]))
    # the reference's public fields (Band-Edge Filter.cs:19-26): design parameters, and phase / freq writable between calls
    assert (g1.sps, g1.rolloff, g1.filterSize, g1.bandwidth) == (4.0, 0.35, 40, 0.02)
    assert (g1.phase, g1.freq) == o1.state
    g1.phase, g1.freq = 1.25, -0.002
    o1.state = (1.25, -0.002)
    assert (g1.phase, g1.freq) == (np.float32(1.25), np.float32(-0.002))
    assert _close(g1.Process(x[1]), o1.Process(x[1]))
    assert gpu.CostasLoopQpsk.GetSign(0.0, -1e-30) == (1.0, -1.0)            # CostasLoopQpsk.cs:52-56
    assert gpu.QPSKModulator(10_000_000, 5_000_000).baudRate == 1_250_000    # QPSKModulator.cs:34


@pytest.mark.parametrize("size", [40, 16, 8, 48, 10, 13, 9, 23, 31, 55, 33, 52])
def test_fll_two_warp_kernel_sizes_and_chunking(gpu, orc, size):
    """8 <= N <= 55 takes the two-warp kernel (csrc/fll_duo.cu; N % 8 != 0 adds the scalar-tail stages): odd chunk lengths exercise the partial last batch,
    the warm-up from the carried ring and the flush bookkeeping; outputs and state must stay bit-identical."""
    x, _ = _qpsk_burst(orc, 900, sps=4, alpha=0.35, cfo=0.03, noise=0.05, seed=size)
    want_f = orc.FLLBandEdgeFilter(4.0, 0.35, size, 0.05)
    got_f = gpu.FLLBandEdgeFilter(4.0, 0.35, size, 0.05)
    cuts = [0, 2, 2 * 4, 2 * 9, 2 * 28, 2 * 61, 2 * 62, 2 * 200, 2 * 777, x.size]
    for a, b in zip(cuts[:-1], cuts[1:]):
        want = want_f.Process(x[a:b])
        got = got_f.Process(x[a:b])
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (size, a, b)
    assert got_f.state == want_f.state


@pytest.mark.parametrize("channels,size", [(700, 40), (1500, 40), (1500, 13)])
def test_fll_many_channels_identical_streams(gpu, orc, channels, size):
    """Every channel gets the same samples: all rows of the batched output must equal the oracle's single stream bit
    for bit.  Loads every SM with chain / side warp pairs (one pair per CTA below 1280 streams, four above), which is
    where a hand-over or ordering bug between the two warps would show."""
    x, _ = _qpsk_burst(orc, 1200, sps=4, alpha=0.35, cfo=0.02, noise=0.05, seed=3)
    X = np.ascontiguousarray(np.broadcast_to(x, (channels, x.size)))
    f = gpu.FLLBandEdgeFilter(4.0, 0.35, size, 0.05, channels=channels)
    o = orc.FLLBandEdgeFilter(4.0, 0.35, size, 0.05)
    cut = 2 * 1111
    for a, b in [(0, cut), (cut, x.size)]:
        want = o.Process(x[a:b])
        got = f.Process(np.ascontiguousarray(X[:, a:b]))
        assert np.array_equal(got.view(np.uint32), np.broadcast_to(want.view(np.uint32), got.shape))


@pytest.mark.parametrize("sps,size,L", [(0.5, 40, 300), (1.0, 10, 1), (3.0, 24, 2), (4.0, 40, 3), (2.0, 55, 5), (16.0, 8, 77)])
def test_fll_two_warp_kernel_short_calls_and_odd_rates(gpu, orc, sps, size, L):
    """Calls shorter than one hand-over batch (1..5 samples), repeated, and symbol rates that make the frequency limit
    large (sps 0.5: +-8 pi per sample, the phase wraps on most samples)."""
    x, _ = _qpsk_burst(orc, 400, sps=4, alpha=0.35, cfo=0.05, noise=0.05, seed=int(10 * sps) + size)
    want_f = orc.FLLBandEdgeFilter(sps, 0.35, size, 0.2)
    got_f = gpu.FLLBandEdgeFilter(sps, 0.35, size, 0.2)
    pos = 0
    for k in range(12):
        n = L if k % 3 else L + 4 * k
        want = want_f.Process(x[pos:pos + 2 * n])
        got = got_f.Process(x[pos:pos + 2 * n])
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (k, n)
        pos += 2 * n
    assert got_f.state == want_f.state


def test_fll_phase_wrap_and_wild_state(gpu, orc):
    """A large loop bandwidth drives the phase past +-2*pi every few samples (the wrap path, Band-Edge Filter.cs:185-189);
    a caller-set phase far outside the loop's range must take the generic kernel and still match."""
    x, _ = _qpsk_burst(orc, 600, sps=2, alpha=0.5, cfo=0.2, noise=0.02, seed=5)
    for state in [None, (3.0e4, 0.5), (-7.0, -3.0)]:
        want_f = orc.FLLBandEdgeFilter(2.0, 0.5, 40, 0.5)
        got_f = gpu.FLLBandEdgeFilter(2.0, 0.5, 40, 0.5)
        if state is not None:
            want_f.state = state
            got_f.state = state
        for a, b in [(0, 2 * 301), (2 * 301, x.size)]:
            want = want_f.Process(x[a:b])
            got = got_f.Process(x[a:b])
            assert _close(got, want)
            assert np.mean(got.view(np.uint32) == want.view(np.uint32)) > 0.999
        pw, fw = want_f.state
        pg, fg = got_f.state
        assert abs(pw - pg) <= 1e-4 * max(1.0, abs(pw)) and abs(fw - fg) <= 1e-5 * max(abs(fw), 1e-3)


def test_fll_errors(gpu, orc):
    for mod in (gpu, orc):
        for args in [(0.0, 0.5, 10, 0.1), (2.0, -0.1, 10, 0.1), (2.0, 1.5, 10, 0.1), (2.0, 0.5, 0, 0.1), (2.0, 0.5, 10, 0.0)]:
            with pytest.raises(mod.ArgumentOutOfRangeException):
                mod.FLLBandEdgeFilter(*args)
        f = mod.FLLBandEdgeFilter(2.0, 0.5, 10, 0.1)
        with pytest.raises(mod.ArgumentException):
            f.Process(np.zeros(3, np.float32))
        with pytest.raises(mod.ArgumentException):
            f.Process(np.zeros(4, np.float32), out_len=2)


@pytest.mark.parametrize("sps,bw", [(2, 1e-4), (4, 1e-3), (4, 0.05), (30, 2e-9), (3, 0.01)])
def test_mm_matches_oracle_chunked(gpu, orc, sps, bw):
    x, _ = _qpsk_burst(orc, 1200, sps=sps, noise=0.01, seed=sps)
    mf = orc.ComplexFIRFilter(orc.real_taps_to_iq(orc.RRCFilter.generateCoefficents(10, 0.35, sps * 1000, 1000))).Filter(x)
    kp, ki = orc.mm_gains_from_bw(bw)
    kpg, kig = gpu.mm_gains_from_bw(bw)
    assert (kp, ki) == (kpg, kig)
    want_m = orc.MuellerMuller(float(sps), kp, ki)
    got_m = gpu.MuellerMuller(float(sps), kp, ki)
    cuts = [0, 2, 4, 10, 2 * 101, 2 * 999, 2 * 1000, mf.size]
    for a, b in zip(cuts[:-1], cuts[1:]):
        want = want_m.Process(mf[a:b])
        got = got_m.Process(mf[a:b])
        assert got.shape == want.shape
        assert _close(got, want)
        ws, gs = want_m.state, got_m.state
        assert ws["baseIndex"] == gs["baseIndex"] and ws["queued"] == gs["queued"]
        assert abs(ws["mu"] - gs["mu"]) < 1e-9 and abs(ws["ncoIntegral"] - gs["ncoIntegral"]) < 1e-12
    # chunk-invariance (MuellerMuller.cs:122-133): one shot == chunked
    one = gpu.MuellerMuller(float(sps), kp, ki).Process(mf)
    ref = orc.MuellerMuller(float(sps), kp, ki).Process(mf)
    assert _close(one, ref)


def test_mm_first_symbol_and_small_output(gpu, orc):
    """SURVEY §4.5: first symbol emitted without TED update at baseIndex=1, mu=0; a too-small output
    span stops early and keeps the rest queued (the integrator quirk at :83/:101 included)."""
    x, _ = _qpsk_burst(orc, 400, sps=4, seed=9)
    mf = orc.ComplexFIRFilter(orc.real_taps_to_iq(orc.RRCFilter.generateCoefficents(10, 0.35, 4000, 1000))).Filter(x)
    kp, ki = orc.mm_gains_from_bw(0.01)
    g, o = gpu.MuellerMuller(4.0, kp, ki), orc.MuellerMuller(4.0, kp, ki)
    got, want = g.Process(mf[:40], cap_floats=5), o.Process(mf[:40], cap_floats=5)
    assert got.shape == want.shape == (4,)     # cap 5 floats -> 2 symbols (o+1 >= Length breaks at o=4)
    assert _close(got, want)
    assert g.state == pytest.approx(o.state)
    got, want = g.Process(mf[40:]), o.Process(mf[40:])
    assert got.shape == want.shape and _close(got, want)
    # with mu == 0 the interpolator returns x[baseIndex] exactly
    g2 = gpu.MuellerMuller(4.0, kp, ki)
    first = g2.Process(mf[:16])
    assert np.array_equal(first[:2], mf[2:4])


def test_mm_batch(gpu, orc):
    C = 4
    kp, ki = orc.mm_gains_from_bw(1e-3)
    mfs = []
    for c in range(C):
        x, _ = _qpsk_burst(orc, 500, sps=4, noise=0.02, seed=70 + c)
        mfs.append(orc.ComplexFIRFilter(orc.real_taps_to_iq(orc.RRCFilter.generateCoefficents(10, 0.35, 4000, 1000))).Filter(x))
    x = np.stack(mfs)
    got = gpu.MuellerMuller(4.0, kp, ki, channels=C).Process(x)
    for c in range(C):
        want = orc.MuellerMuller(4.0, kp, ki).Process(x[c])
        assert got[c].shape == want.shape and _close(got[c], want)


@pytest.mark.parametrize("fs,bw", [(5_000_000.0, 5_000_000.0 / 120), (333333.0, 33333.3), (750000.0, 750000.0 / 130)])
def test_costas_matches_oracle(gpu, orc, fs, bw):
    rng = np.random.default_rng(3)
    n = 3000
    sym = (rng.choice([-1, 1], n) + 1j * rng.choice([-1, 1], n)) / np.sqrt(2)
    z = sym * np.exp(1j * (0.4 + 2 * np.pi * 2e-4 * np.arange(n))) + 0.03 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    x = np.empty(2 * n, np.float32)
    x[0::2], x[1::2] = z.real, z.imag
    g, o = gpu.CostasLoopQpsk(fs, bw), orc.CostasLoopQpsk(fs, bw)
    for a, b in [(0, 2), (2, 2000), (2000, 2 * n)]:
        want, got = o.Process(x[a:b]), g.Process(x[a:b])
        assert _close(got, want)
    tw, fw = o.GetState()
    tg, fg = g.GetState()
    assert abs(tw - tg) < 1e-9 and abs(fw - fg) < 1e-12
    for mod in (gpu, orc):
        c = mod.CostasLoopQpsk(fs, bw)
        with pytest.raises(mod.ArgumentException):
            c.Process(np.zeros(3, np.float32))
        with pytest.raises(mod.ArgumentException):
            c.Process(np.zeros(4, np.float32), out_len=2)


def test_fll_large_batch_kernel_choice_and_far_phase(gpu, orc):
    """From 5120 streams the two-lanes-per-stream kernel (fll_pair_kernel) serves the FLL.  Its sin/cos is the |phase| < 64
    form, so a caller-set phase beyond 32 goes through the two-warp kernel (fll_duo_kernel) for one call (which leaves the
    phase wrapped); both calls, and the loop state after them, must be the oracle's bit for bit."""
    C, L = 5200, 300
    rng = np.random.default_rng(21)
    x = (0.4 * rng.standard_normal((C, 2 * L))).astype(np.float32)
    g = gpu.FLLBandEdgeFilter(2.0, 0.4, 40, 0.02, channels=C)
    ph = np.zeros(C, np.float32)
    fr = np.zeros(C, np.float32)
    probe = [0, 1, 31, 32, 2600, C - 1]
    ph[probe] = np.array([50.0, -37.5, 0.3, 6.5, 1000.25, -63.0], np.float32)
    fr[probe] = np.array([0.1, -0.2, 0.0, 0.5, 0.01, -0.4], np.float32)
    g.state = (ph, fr)
    outs = [g.Process(x), g.Process(x[:, ::-1].copy())]        # first call: duo kernel (far phase); second: pair kernel
    gp, gf = g.state
    for c in probe + [7, 4000]:
        o = orc.FLLBandEdgeFilter(2.0, 0.4, 40, 0.02)
        o.state = (float(ph[c]), float(fr[c]))
        w0 = o.Process(x[c])
        w1 = o.Process(x[c, ::-1].copy())
        assert np.array_equal(outs[0][c].view(np.uint32), w0.view(np.uint32)), c
        assert np.array_equal(outs[1][c].view(np.uint32), w1.view(np.uint32)), c
        op, of = o.state
        assert np.float32(op) == gp[c] and np.float32(of) == gf[c], c
