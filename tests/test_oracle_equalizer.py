"""CPU: the blind CMA equalizer (not in the reference; spec in include/qpskcuda.h).  Its two CPU restatements
(tests/cma_oracle.py) must agree bit for bit; the oracle demodulator with the stage must equal the CPU oracle's
QPSKDeModulator while the stage is off, and must earn its place on a multipath channel that the reference receive chain
cannot decode."""
import numpy as np
import pytest

from cma_oracle import CmaBatch, CmaScalar, EqArgumentError, EqDemod

TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"
FS, RS = 10_000_000, 5_000_000            # sps 2, 21-tap RRC matched filter: the bench geometry
ALPHA = float(np.float32(0.4))
SPAN = 10

# The frozen multipath channel: a second path of gain 0.55+0.55j (|g| = 0.78) one symbol (two samples) late, AWGN at
# -25 dBFS, the two unstable LOs of the channel simulator (100 MHz, 1 ppm each).  Its complex echo closes the eye of the
# hard decisions: the chain without an equalizer gets about a third of the bits wrong.
FROZEN = dict(path_gains_iq=(1.0, 0.0, 0.55, 0.55), path_delays=(0, 2), noise_dbfs=-25.0, lo_hz=100e6, ppm=1.0)
FROZEN_EQ = dict(n_taps=11, mu=0.01)      # mu chosen on this channel: converges within the first burst
N_PAYLOAD, BURSTS = 256, 6


def frozen_frame(orc, seed: int):
    """(tx samples of one frame, the frame's bits as uint8 0/1 incl. the TSC): frames follow each other back to back."""
    pay = np.random.default_rng(seed).integers(0, 256, N_PAYLOAD, dtype=np.uint8).tobytes()
    tx = orc.QPSKModulator(FS, RS, ALPHA, SPAN, tsc=TSC).ModulateBytes(pay, b"S", b"E")
    ref = np.frombuffer((TSC + orc.BitPacker.BytesToBitString(b"S" + pay + b"E")).encode(), np.uint8) - ord("0")
    return tx, ref


def burst_errors(bits: np.ndarray, ref: np.ndarray, max_offset: int = 80):
    """Bit errors of one burst's demodulated bits (uint8 0/1, differential decoding, no TSC strip) against the frame.
    The bits are aligned with the frame by the best of the first `max_offset` offsets (the symbols before the frame are
    the previous frame's tail); the first dibit is skipped (its differential reference is the idle gap before the frame)
    and the last 16 bits (END marker and the symbols an equalizer's group delay carries into the next call).  Bits that
    did not arrive count as errors.  Returns (errors, bits counted)."""
    want = ref[2:ref.size - 16]
    best = None
    for o in range(max_offset):
        got = bits[o:o + want.size]
        e = int((got != want[:got.size]).sum()) + (want.size - got.size)
        best = e if best is None else min(best, e)
    return best, want.size


def frozen_channel_ber(orc, eq, channel: int = 0, seed: int = 5):
    """Per-burst errors of the oracle demodulator (differential, no TSC strip) on the frozen channel."""
    tx, ref = frozen_frame(orc, seed)
    n = tx.size // 2
    f = FROZEN
    txo = orc.NCO(f["lo_hz"], FS, f["ppm"], seed=seed, stream=4 * channel)
    rxo = orc.NCO(f["lo_hz"], FS, f["ppm"], seed=seed, stream=4 * channel + 1)
    if eq:
        dem = EqDemod(orc, FS, RS, ALPHA, SPAN)
        dem.set_equalizer(FROZEN_EQ["n_taps"], FROZEN_EQ["mu"])
        demod = lambda y: dem.DeModulate(y)[0]                  # noqa: E731
    else:
        demod = orc.QPSKDeModulator(FS, RS, ALPHA, SPAN).DeModulate
    out = []
    for b in range(BURSTS):
        mp = orc.multipath(tx, f["path_gains_iq"], f["path_delays"])
        nz = orc.noise_iq(f["noise_dbfs"], n, seed, 4 * channel + 2, b * n)
        y = orc.channel_apply(txo, rxo, 1, mp, nz)
        bits = np.frombuffer(demod(y).encode(), np.uint8) - ord("0")
        out.append(burst_errors(bits, ref))
    return out


@pytest.mark.parametrize("n_taps", [1, 2, 7, 11, 64])
@pytest.mark.parametrize("mu", [0.0, 1e-3, 0.03])
def test_batch_and_scalar_restatements_agree(orc, n_taps, mu):
    C = 3
    x = np.stack([orc.fill_uniform(n_taps, 11 + c, 0, 2 * 240) * np.float32(1.4) for c in range(C)]).astype(np.float32)
    b = CmaBatch(n_taps, mu, 1.0, C)
    got = b.process(x)
    for c in range(C):
        s = CmaScalar(n_taps, mu)
        want = s.Process(x[c])
        assert np.array_equal(got[c].view(np.uint32), want.view(np.uint32)), c
        assert np.array_equal(b.taps[c].view(np.uint32), s.taps.view(np.uint32)), c
    if mu > 0:
        assert not np.array_equal(b.taps, CmaBatch(n_taps, mu, 1.0, C).taps)    # the taps adapt


def test_batch_ragged_counts_and_discard(orc):
    C, N = 6, 7
    x = np.stack([orc.fill_uniform(2, c, 0, 2 * 50) for c in range(C)]).astype(np.float32)
    lengths = [50, 0, 1, 3, 4, 29]
    b = CmaBatch(N, 0.05, 1.0, C)
    got = b.process(x, lengths, drop=True)
    for c in range(C):
        want = CmaScalar(N, 0.05).Process(x[c, : 2 * lengths[c]])
        assert np.array_equal(got[c].view(np.uint32), want[2 * 3:].view(np.uint32)), c     # (N-1)//2 = 3 discarded
    assert b.drop.tolist() == [0, 3, 2, 0, 0, 0]
    more = b.process(x[:, :20], drop=True)                               # the rest of the discard, then nothing
    assert [m.size for m in more] == [20, 14, 16, 20, 20, 20]


@pytest.mark.parametrize("n_taps", [2, 11, 64])
def test_chunking_is_bit_exact(orc, n_taps):
    x = orc.fill_uniform(3, n_taps, 0, 2 * 600)[None, :]
    want = CmaBatch(n_taps, 0.02, 1.5).process(x)[0]
    rng = np.random.default_rng(n_taps)
    for _ in range(2):
        cuts = np.sort(rng.choice(np.arange(1, 600), 6, replace=False)) * 2
        e = CmaBatch(n_taps, 0.02, 1.5)
        got = np.concatenate([e.process(p)[0] for p in np.split(x, cuts, axis=1)])
        assert np.array_equal(want.view(np.uint32), got.view(np.uint32))


def test_taps_reset_and_arguments(orc):
    e = CmaBatch(7, 0.05)
    spike = np.zeros((1, 14), np.float32)
    spike[0, 2 * 3] = 1.0
    assert np.array_equal(e.taps, spike)                                 # w[(N-1)/2] = 1
    x = orc.fill_uniform(4, 0, 0, 400)[None, :]
    y0 = e.process(x)[0]
    assert not np.array_equal(e.taps, spike)
    e.reset()
    assert np.array_equal(e.taps, spike)
    assert np.array_equal(e.process(x)[0].view(np.uint32), y0.view(np.uint32))
    for args, status in [((7, -0.1), -3), ((7, 0.1, 0.0), -3), ((7, float("nan")), -3), ((7, float("inf")), -3),
                         ((0, 0.1), -7), ((65, 0.1), -7)]:
        with pytest.raises(EqArgumentError) as ei:
            CmaBatch(*args)
        assert ei.value.status == status


@pytest.mark.parametrize("use_fll", [False, True])
@pytest.mark.parametrize("tsc", [TSC, None])
def test_oracle_demod_wiring_equals_the_oracle_without_the_stage(orc, use_fll, tsc):
    """EqDemod is the CPU oracle's blocks wired as its QPSKDeModulator wires them: with the stage off (and with the identity
    stage: one tap, mu 0) bits, payloads and constellation equal oracle.QPSKDeModulator's bit for bit."""
    C = 3
    rx = []
    for c in range(C):
        tx, _ = frozen_frame(orc, 3 + c)
        txo, rxo = orc.NCO(100e6, FS, 1, seed=9, stream=4 * c), orc.NCO(100e6, FS, 1, seed=9, stream=4 * c + 1)
        mp = orc.multipath(np.concatenate([tx] * 3), (1.0, 0.0, 0.12, 0.08), (0, 3))
        rx.append(orc.channel_apply(txo, rxo, 1, mp, orc.noise_iq(-40.0, mp.size // 2, 9, 4 * c + 2)))
    rx = np.stack(rx)
    bursts = np.split(rx, [2 * 1500, 2 * 4000], axis=1)
    kw = dict(tsc=tsc, use_fll=use_fll)
    for eq in (None, (1, 0.0)):
        mk = lambda: EqDemod(orc, FS, RS, ALPHA, SPAN, channels=C, **kw)  # noqa: E731
        d_bits, d_bytes, d_cons = mk(), mk(), mk()
        if eq:
            for d in (d_bits, d_bytes, d_cons):
                d.set_equalizer(*eq)
        o = {k: [orc.QPSKDeModulator(FS, RS, ALPHA, SPAN, **kw) for _ in range(C)] for k in ("bits", "bytes", "cons")}
        frames = 0
        for b in bursts:
            b = np.ascontiguousarray(b)
            bits, pays, cons = d_bits.DeModulate(b), d_bytes.DeModulateBytes(b, b"S", b"E"), d_cons.deModulateConstellation(b)
            for c in range(C):
                assert bits[c] == o["bits"][c].DeModulate(b[c]), (eq, c)
                w = o["bytes"][c].DeModulateBytes(b[c], b"S", b"E", cap=1 << 16)
                assert pays[c] == w, (eq, c)
                frames += len(w) > 0
                assert np.array_equal(cons[c].view(np.uint32), o["cons"][c].deModulateConstellation(b[c]).view(np.uint32))
        assert frames > 0


def test_oracle_demod_equalizer_chunking(orc):
    """The stage's group delay is absorbed once per stream: any chunking of the samples gives the same bit stream."""
    tx, _ = frozen_frame(orc, 6)
    f = FROZEN
    x = np.concatenate([orc.multipath(tx, f["path_gains_iq"], f["path_delays"])] * 2)
    one = EqDemod(orc, FS, RS, ALPHA, SPAN)
    one.set_equalizer(11, 0.01)
    want = one.DeModulate(x)[0]
    parts = EqDemod(orc, FS, RS, ALPHA, SPAN)
    parts.set_equalizer(11, 0.01)
    cuts = [0, 2 * 301, 2 * 1700, 2 * 1701, 2 * 3999, x.size]
    got = "".join(parts.DeModulate(x[a:b])[0] for a, b in zip(cuts[:-1], cuts[1:]))
    assert got == want
    assert np.array_equal(one.equalizer_taps(), parts.equalizer_taps())


def test_equalizer_recovers_the_frozen_multipath_channel(orc):
    off = frozen_channel_ber(orc, eq=False)
    on = frozen_channel_ber(orc, eq=True)
    e_off, n_off = map(sum, zip(*off[1:]))
    e_on, n_on = map(sum, zip(*on[1:]))
    assert e_off / n_off >= 1e-2, off          # the reference chain cannot decode this channel
    assert e_on / n_on <= 1e-3, on             # with the equalizer it does, after the first burst
