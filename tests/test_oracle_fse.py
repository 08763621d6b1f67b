"""CPU: the fractionally spaced (T/sps) form of the blind CMA equalizer and the demodulator's fractionally spaced stage
(spec in include/qpskcuda.h).  The two CPU restatements (tests/fse_oracle.py) must agree bit for bit at every update
stride; the stage ahead of Mueller-Muller must be transparent as a spike with mu 0, and must earn its place against the
symbol-spaced stage on the frozen multipath channel."""
import numpy as np
import pytest

from cma_oracle import CmaBatch, EqArgumentError
from fse_oracle import FseBatch, FseDemod, FseScalar
from test_oracle_equalizer import ALPHA, BURSTS, FROZEN, FROZEN_EQ, FS, RS, SPAN, TSC, burst_errors, frozen_frame

U32 = np.uint32
FROZEN_FSE = dict(n_taps=21, mu=0.005)    # 21 taps at T/2 span the same +-5 symbols as the 11-tap symbol-spaced stage

# Draws d of the frozen channel: payload / LO / noise seed 5 + d, LO and noise streams of channel d % 4.
DRAWS = list(range(24))
# The draws on which the chain loses a late burst (2-6) with no second path and no equalizer at all, FLL off: the LO model
# alone costs these bursts, so they say nothing about equalization (test_lo_draws_lose_late_bursts_without_multipath).
LO_DRAWS = [7, 15, 17, 20, 23]


def draw_bursts(orc, draws, gains=FROZEN["path_gains_iq"]):
    """BURSTS blocks [len(draws), n] of the frozen channel, one row per draw, and each draw's reference bits."""
    f = FROZEN
    frames = [frozen_frame(orc, 5 + d) for d in draws]
    txo = [orc.NCO(f["lo_hz"], FS, f["ppm"], seed=5 + d, stream=4 * (d % 4)) for d in draws]
    rxo = [orc.NCO(f["lo_hz"], FS, f["ppm"], seed=5 + d, stream=4 * (d % 4) + 1) for d in draws]
    out = []
    for b in range(BURSTS):
        rows = []
        for i, d in enumerate(draws):
            tx = frames[i][0]
            n = tx.size // 2
            nz = orc.noise_iq(f["noise_dbfs"], n, 5 + d, 4 * (d % 4) + 2, b * n)
            rows.append(orc.channel_apply(txo[i], rxo[i], 1, orc.multipath(tx, gains, f["path_delays"]), nz))
        out.append(np.stack(rows))
    return out, [r for _, r in frames]


def burst_table(orc, dem, bursts, refs):
    """errors [draw, burst] of FseDemod `dem` (one channel per draw)"""
    errs = np.zeros((len(refs), len(bursts)), np.int64)
    for b, rx in enumerate(bursts):
        for i, bits in enumerate(dem.DeModulate(rx)):
            errs[i, b] = burst_errors(np.frombuffer(bits.encode(), np.uint8) - ord("0"), refs[i])[0]
    return errs


def stage_errors(orc, bursts, refs, kind, use_fll=False):
    dem = FseDemod(orc, FS, RS, ALPHA, SPAN, channels=len(refs), use_fll=use_fll)
    if kind == "eq":
        dem.set_equalizer(FROZEN_EQ["n_taps"], FROZEN_EQ["mu"])
    elif kind == "fse":
        dem.set_fractional_equalizer(FROZEN_FSE["n_taps"], FROZEN_FSE["mu"])
    return burst_table(orc, dem, bursts, refs)


# ---- the block ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sps", [2, 3, 4])
@pytest.mark.parametrize("n_taps", [1, 2, 11, 21, 64])
@pytest.mark.parametrize("mu", [0.0, 1e-3, 0.03])
def test_batch_and_scalar_restatements_agree(orc, sps, n_taps, mu):
    C = 3
    x = np.stack([orc.fill_uniform(n_taps, 21 + c, 0, 2 * 240) * np.float32(1.4) for c in range(C)]).astype(np.float32)
    b = FseBatch(n_taps, mu, 1.0, C, sps=sps)
    got = b.process(x)
    for c in range(C):
        s = FseScalar(n_taps, mu, sps=sps)
        want = s.Process(x[c])
        assert np.array_equal(got[c].view(U32), want.view(U32)), c
        assert np.array_equal(b.taps[c].view(U32), s.taps.view(U32)), c
    if mu > 0:
        # the taps adapt, and on every sps-th sample only: not as the symbol-spaced equalizer does on the same input
        assert not np.array_equal(b.taps, FseBatch(n_taps, mu, 1.0, C, sps=sps).taps)
        s1 = CmaBatch(n_taps, mu, 1.0, C)
        s1.process(x)
        assert not np.array_equal(b.taps, s1.taps)


def test_stride_one_is_the_symbol_spaced_equalizer(orc):
    x = orc.fill_uniform(5, 1, 0, 2 * 300)[None, :]
    a, b = CmaBatch(11, 0.02), FseBatch(11, 0.02, sps=1)
    assert np.array_equal(a.process(x)[0].view(U32), b.process(x)[0].view(U32))


@pytest.mark.parametrize("sps", [2, 4, 3])
@pytest.mark.parametrize("n_taps", [2, 21])
def test_chunking_is_bit_exact(orc, sps, n_taps):
    """Odd cut points put cuts in the middle of a symbol: the phase of the update stride must carry over."""
    L = 601
    x = orc.fill_uniform(3, n_taps, 0, 2 * L)[None, :]
    one = FseBatch(n_taps, 0.02, 1.5, sps=sps)
    want = one.process(x, drop=True)[0]
    for cuts in ([1, 2, 7, 300, 301, 599], [3, 5, 9, 11, 13, 500]):
        e = FseBatch(n_taps, 0.02, 1.5, sps=sps)
        got = np.concatenate([e.process(p, drop=True)[0] for p in np.split(x, np.array(cuts) * 2, axis=1)])
        assert np.array_equal(want.view(U32), got.view(U32)), cuts
        assert np.array_equal(e.taps.view(U32), one.taps.view(U32))
        assert e.phase.tolist() == [L % sps]


@pytest.mark.parametrize("sps", [2, 4])
def test_batch_ragged_counts_and_discard(orc, sps):
    C, N = 6, 7
    x = np.stack([orc.fill_uniform(2, c, 0, 2 * 50) for c in range(C)]).astype(np.float32)
    lengths = [50, 0, 1, 3, 4, 29]
    b = FseBatch(N, 0.05, 1.0, C, sps=sps)
    got = b.process(x, lengths, drop=True)
    scal = [FseScalar(N, 0.05, sps=sps) for _ in range(C)]
    for c in range(C):
        want = scal[c].Process(x[c, : 2 * lengths[c]])
        assert np.array_equal(got[c].view(U32), want[2 * 3:].view(U32)), c     # (N-1)//2 = 3 discarded
    assert b.drop.tolist() == [0, 3, 2, 0, 0, 0]
    assert b.phase.tolist() == [n % sps for n in lengths]
    # every channel goes on from its own count: the phase differs between channels
    x2 = np.stack([orc.fill_uniform(8, c, 0, 2 * 21) for c in range(C)]).astype(np.float32)
    more = b.process(x2, drop=True)
    assert [m.size for m in more] == [42, 36, 38, 42, 42, 42]
    for c in range(C):
        want = scal[c].Process(x2[c])
        assert np.array_equal(more[c].view(U32), want[want.size - more[c].size:].view(U32)), c
        assert np.array_equal(b.taps[c].view(U32), scal[c].taps.view(U32)), c


def test_taps_reset_and_arguments(orc):
    e = FseBatch(7, 0.05, sps=2)
    x = orc.fill_uniform(4, 0, 0, 2 * 201)[None, :]
    y0 = e.process(x)[0]
    assert e.phase.tolist() == [1]
    e.reset()
    assert e.phase.tolist() == [0]
    assert np.array_equal(e.process(x)[0].view(U32), y0.view(U32))
    for args, status in [((7, -0.1), -3), ((7, 0.1, 0.0), -3), ((7, float("nan")), -3), ((0, 0.1), -7), ((65, 0.1), -7)]:
        with pytest.raises(EqArgumentError) as ei:
            FseBatch(*args, sps=2)
        assert ei.value.status == status
    for sps in (0, 9, -1):
        with pytest.raises(EqArgumentError) as ei:
            FseBatch(7, 0.1, sps=sps)
        assert ei.value.status == -7
    # the demodulator stage needs an integer rate of 2..8 samples per symbol; n_taps 0 is always accepted (off)
    for fs, rs in ((10_000_000, 3_000_000), (5_000_000, 5_000_000), (9_000_000, 1_000_000)):
        d = FseDemod(orc, fs, rs, ALPHA, SPAN)
        with pytest.raises(EqArgumentError) as ei:
            d.set_fractional_equalizer(11, float("nan"))
        assert ei.value.status == -7
        d.set_fractional_equalizer(0, 0.0)
    d = FseDemod(orc, 8_000_000, 1_000_000, ALPHA, SPAN)
    d.set_fractional_equalizer(11, 0.01)
    assert d.fse.sps == 8
    with pytest.raises(EqArgumentError) as ei:
        d.set_fractional_equalizer(11, -1.0)
    assert ei.value.status == -3


# ---- the demodulator stage -----------------------------------------------------------------------------------------------
def _bench_like_bursts(orc, C):
    rx = []
    for c in range(C):
        tx, _ = frozen_frame(orc, 3 + c)
        txo, rxo = orc.NCO(100e6, FS, 1, seed=9, stream=4 * c), orc.NCO(100e6, FS, 1, seed=9, stream=4 * c + 1)
        mp = orc.multipath(np.concatenate([tx] * 3), (1.0, 0.0, 0.12, 0.08), (0, 3))
        rx.append(orc.channel_apply(txo, rxo, 1, mp, orc.noise_iq(-40.0, mp.size // 2, 9, 4 * c + 2)))
    return np.split(np.stack(rx), [2 * 1501, 2 * 4000], axis=1)       # odd cut: mid-symbol


@pytest.mark.parametrize("use_fll", [False, True])
@pytest.mark.parametrize("tsc", [TSC, None])
def test_one_tap_stage_equals_the_oracle(orc, use_fll, tsc):
    """One tap, mu 0: the identity with no delay.  Bits, payloads and constellation equal oracle.QPSKDeModulator's bit
    for bit in every call."""
    C = 3
    kw = dict(tsc=tsc, use_fll=use_fll)
    mk = lambda: FseDemod(orc, FS, RS, ALPHA, SPAN, channels=C, **kw)  # noqa: E731
    d_bits, d_bytes, d_cons = mk(), mk(), mk()
    for d in (d_bits, d_bytes, d_cons):
        d.set_fractional_equalizer(1, 0.0)
    o = {k: [orc.QPSKDeModulator(FS, RS, ALPHA, SPAN, **kw) for _ in range(C)] for k in ("bits", "bytes", "cons")}
    frames = 0
    for b in _bench_like_bursts(orc, C):
        b = np.ascontiguousarray(b)
        bits, pays, cons = d_bits.DeModulate(b), d_bytes.DeModulateBytes(b, b"S", b"E"), d_cons.deModulateConstellation(b)
        for c in range(C):
            assert bits[c] == o["bits"][c].DeModulate(b[c]), c
            w = o["bytes"][c].DeModulateBytes(b[c], b"S", b"E", cap=1 << 16)
            assert pays[c] == w, c
            frames += len(w) > 0
            assert np.array_equal(cons[c].view(U32), o["cons"][c].deModulateConstellation(b[c]).view(U32))
    assert frames > 0


@pytest.mark.parametrize("use_fll", [False, True])
@pytest.mark.parametrize("tsc", [TSC, None])
def test_spike_stage_with_mu_zero_equals_the_oracle_stream(orc, use_fll, tsc):
    """A 21-tap spike with mu 0 delays the matched-filter output by 10 samples, and the discard takes the delay back out:
    Mueller-Muller sees the oracle's sample stream, the last 10 samples of a call in the next.  So the symbol stream, and
    without a TSC the bit stream, are the oracle's, each call's share ending at most a few symbols earlier.  (The TSC strip
    and the framer's marker hunt look at each call's bits on their own, so what they give depends on where a call ends;
    the one-tap test covers them call by call.)"""
    C = 3
    kw = dict(tsc=tsc, use_fll=use_fll)
    mk = lambda: FseDemod(orc, FS, RS, ALPHA, SPAN, channels=C, **kw)  # noqa: E731
    d_bits, d_cons = mk(), mk()
    for d in (d_bits, d_cons):
        d.set_fractional_equalizer(21, 0.0)
    o = {k: [orc.QPSKDeModulator(FS, RS, ALPHA, SPAN, **kw) for _ in range(C)] for k in ("bits", "cons")}
    got = {k: [[] for _ in range(C)] for k in o}
    want = {k: [[] for _ in range(C)] for k in o}
    for b in _bench_like_bursts(orc, C):
        b = np.ascontiguousarray(b)
        bits, cons = d_bits.DeModulate(b), d_cons.deModulateConstellation(b)
        for c in range(C):
            got["bits"][c].append(bits[c])
            got["cons"][c].append(cons[c])
            want["bits"][c].append(o["bits"][c].DeModulate(b[c]))
            want["cons"][c].append(o["cons"][c].deModulateConstellation(b[c]))
    for c in range(C):
        g, w = np.concatenate(got["cons"][c]), np.concatenate(want["cons"][c])
        assert np.array_equal(g.view(U32), w[: g.size].view(U32)) and w.size - g.size <= 16, c
        if tsc is None:
            g, w = "".join(got["bits"][c]), "".join(want["bits"][c])
            assert w.startswith(g) and len(w) - len(g) <= 16, (c, len(w) - len(g))


def test_oracle_demod_fractional_stage_chunking(orc):
    """The stage's state (taps, window, update phase, discard) carries across calls: any chunking of the samples, cuts in
    the middle of a symbol included, gives the same bit stream."""
    tx, _ = frozen_frame(orc, 6)
    f = FROZEN
    x = np.concatenate([orc.multipath(tx, f["path_gains_iq"], f["path_delays"])] * 2)
    one = FseDemod(orc, FS, RS, ALPHA, SPAN)
    one.set_fractional_equalizer(21, 0.005)
    want = one.DeModulate(x)[0]
    parts = FseDemod(orc, FS, RS, ALPHA, SPAN)
    parts.set_fractional_equalizer(21, 0.005)
    cuts = [0, 2 * 3, 2 * 301, 2 * 1700, 2 * 1703, 2 * 3999, x.size]
    got = "".join(parts.DeModulate(x[a:b])[0] for a, b in zip(cuts[:-1], cuts[1:]))
    assert got == want
    assert np.array_equal(one.fractional_equalizer_taps(), parts.fractional_equalizer_taps())


def test_fractional_stage_recovers_the_frozen_multipath_channel(orc):
    bursts, refs = draw_bursts(orc, [0])                # seed 5, channel 0: the channel of test_oracle_equalizer.py
    errs = stage_errors(orc, bursts, refs, "fse")[0]
    n = burst_errors(np.zeros(0, np.uint8), refs[0])[1]
    assert errs[1:].sum() / (n * (BURSTS - 1)) <= 1e-3, errs


def test_lo_draws_lose_late_bursts_without_multipath(orc):
    """With a single path and no equalizer, the draws of LO_DRAWS (and only those) lose a late burst: the LO model, not
    the echo, costs them."""
    bursts, refs = draw_bursts(orc, DRAWS, gains=(1.0, 0.0, 0.0, 0.0))
    errs = stage_errors(orc, bursts, refs, "off")
    assert [d for d in DRAWS if errs[d, 1:].sum() > 0] == LO_DRAWS, errs


def test_fractional_stage_beats_the_symbol_spaced_stage(orc):
    """Bursts 2-6 of the frozen channel over DRAWS less LO_DRAWS (19 draws).  The restatement gives, FLL off: the T/2 stage
    ahead of Mueller-Muller decodes 16 draws with no error and 702 bit errors in all, the symbol-spaced stage after it 1
    draw and 883 errors (the other three T/2 draws lose a late burst: 8 and 13 after MM slips, 16 in burst 2)."""
    ds = [d for d in DRAWS if d not in LO_DRAWS]
    bursts, refs = draw_bursts(orc, ds)
    fse = stage_errors(orc, bursts, refs, "fse")[:, 1:]
    eq = stage_errors(orc, bursts, refs, "eq")[:, 1:]
    clean_fse, clean_eq = int((fse.sum(1) == 0).sum()), int((eq.sum(1) == 0).sum())
    assert clean_fse >= 15 and clean_eq <= 3, (clean_fse, clean_eq)
    assert fse.sum() <= 0.85 * eq.sum(), (fse.sum(), eq.sum())


def test_fractional_stage_beats_the_symbol_spaced_stage_with_fll(orc):
    """FLL on, all 24 draws, bursts 2-6.  The restatement gives 3896 bit errors with the T/2 stage against 26505 with the
    symbol-spaced one; the T/2 stage decodes bursts 4-6 with no error on 23 draws (all but 14), the symbol-spaced one on
    none."""
    bursts, refs = draw_bursts(orc, DRAWS)
    fse = stage_errors(orc, bursts, refs, "fse", use_fll=True)
    eq = stage_errors(orc, bursts, refs, "eq", use_fll=True)
    assert fse[:, 1:].sum() * 5 <= eq[:, 1:].sum(), (fse[:, 1:].sum(), eq[:, 1:].sum())
    late_fse, late_eq = int((fse[:, 3:].sum(1) == 0).sum()), int((eq[:, 3:].sum(1) == 0).sum())
    assert late_fse >= 22 and late_eq <= 2, (late_fse, late_eq)
