"""CPU: the frame synchronizer's definition (tests/fsync_oracle.py): the pattern is the start of every coded frame, clean
frames are found at their position with every Costas lock phase, the windows decode through the oracle Viterbi decoder to
the frame bits, any chunking gives the same frames, the peak pick beats the lead sidelobes, random data raises few false
alarms at the default threshold, and sync -> Viterbi -> RS recovers payloads on a noisy channel."""
import os
import re

import numpy as np
import pytest

import fec_oracle as V
import fsync_oracle as S
import rs_oracle as R
from fsync_oracle import awgn, frame_bits, stream

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_frame_constants_match_the_header():
    from qpsk_modulator_demodulator_b200 import modem
    hdr = open(os.path.join(ROOT, "include", "qpskcuda.h")).read()
    val = {k: int(v) for k, v in re.findall(r"#define (QPSK_CODED_\w+|QPSK_FSYNC_RHO_DEFAULT) (\d+)", hdr)}
    assert val["QPSK_CODED_LEAD_BITS"] == modem.CODED_LEAD_BITS == S.LEAD_BITS
    assert val["QPSK_CODED_TAIL_BITS"] == modem.CODED_TAIL_BITS == S.TAIL_BITS
    from qpsk_modulator_demodulator_b200 import api
    assert val["QPSK_FSYNC_RHO_DEFAULT"] == api.FSYNC_RHO_DEFAULT == S.RHO_DEFAULT


@pytest.mark.parametrize("start", [b"START", b"\x02", b"\xff\x00\xa5", bytes(range(24))])
def test_pattern_is_the_start_of_every_coded_frame(start):
    pat = S.pattern(start)
    P = S.LEAD_BITS + 8 * len(start)
    assert pat.size == 2 * P and (pat[: 2 * S.LEAD_BITS] == 0).all()
    for pay, end in ((b"\x00" * 3, b"END"), (bytes(range(40)), b""), (b"\xff", b"\x03")):
        coded = V.encode(frame_bits(start, pay, end)[None])[0][0]
        assert coded.size == 2 * S.frame_symbols(len(start), len(pay), len(end))
        assert np.array_equal(coded[: 2 * P], pat)


@pytest.mark.parametrize("differential,rot", [(True, 0), (True, 1), (True, 3), (False, 0), (False, 1), (False, 2),
                                              (False, 3)])
def test_clean_frames_found_at_their_position_and_rotation(differential, rot):
    rng = np.random.default_rng(10 + rot + 4 * differential)
    pays = [rng.integers(0, 256, 20, dtype=np.uint8).tobytes() for _ in range(3)]
    y, pos, fbits = stream(rng, b"START", pays, b"END", [300, 7, 150, 90], differential, rot)
    fs = S.FrameSync(1, differential, b"START", 20, 3)
    got = fs.process(y[None])[0]
    assert [int(i["position"]) for _, i in got] == pos
    for (w, info), b in zip(got, fbits):
        assert int(info["rotation"]) == (0 if differential else rot)
        assert int(info["metric"]) == int(info["energy"]) > 0               # a clean frame matches every soft value
        assert w.size == fs.window
        vit = V.Viterbi(1, differential)
        bits = vit.flush(w[None], w.size)[0]
        assert np.array_equal(bits, b)                                      # bit i is frame bit i


def test_chunking_gives_the_same_frames():
    rng = np.random.default_rng(5)
    Cn = 4
    ys, want = [], []
    for c in range(Cn):
        pays = [rng.integers(0, 256, 4, dtype=np.uint8).tobytes() for _ in range(5)]
        y, pos, _ = stream(rng, b"AB", pays, b"Z", [40, 3, 0, 60, 1, 33], c % 2 == 0)
        ys.append(awgn(rng, y, 6.0))
    n = max(v.size for v in ys)
    Y = np.zeros((Cn, n), np.complex64)
    for c, v in enumerate(ys):
        Y[c, : v.size] = v
    for diff in (True, False):
        whole = S.FrameSync(Cn, diff, b"AB", 4, 1).process(Y)
        assert sum(len(w) for w in whole) >= Cn
        fs = S.FrameSync(Cn, diff, b"AB", 4, 1)
        got = [[] for _ in range(Cn)]
        at = 0
        while at < n:
            step = int(rng.integers(0, 130))
            for c, fr in enumerate(fs.process(Y[:, at: at + step])):
                got[c] += fr
            at += step
        for c in range(Cn):
            assert len(got[c]) == len(whole[c])
            for (wa, ia), (wb, ib) in zip(got[c], whole[c]):
                assert ia == ib and np.array_equal(wa.view(np.uint32), wb.view(np.uint32))


def test_peak_pick_beats_the_lead_sidelobes():
    """the 32 constant lead symbols make the metric ramp up ahead of the frame: at a low threshold the crossing is early,
    and the peak pick still lands on the frame"""
    rng = np.random.default_rng(8)
    y, pos, _ = stream(rng, b"START", [b"\x11" * 8], b"END", [200, 50], False, 2)
    fs = S.FrameSync(1, False, b"START", 8, 3, rho=96)
    s0, s1 = S.soft(y[None], False, fs.scale)
    M, _, E = S.correlate(s0, s1, fs.pat, False)
    first = int(np.nonzero(256 * M[0] >= 96 * E[0])[0][0])
    assert first < pos[0]                                                  # crossing on a sidelobe
    assert [int(i["position"]) for _, i in fs.process(y[None])[0]] == pos


@pytest.mark.parametrize("differential", [False, True])
def test_false_alarms_on_random_data_at_the_default_threshold(differential):
    """random uncoded QPSK (clean and at 3 dB) and pure noise: at most 1 alarm in 2 x 10^5 positions per kind (DESIGN.md
    §3 K15 records the sweep: none in 4.9 x 10^6 per kind)"""
    rng = np.random.default_rng(99 + differential)
    fs = S.FrameSync(50, differential, b"START", 48, 3)
    n = 4000
    q = V.qpsk_symbols(rng.integers(0, 2, (50, 2 * n)), differential)[:, :n]
    for y in (q, awgn(rng, q, 3.0), awgn(rng, np.zeros_like(q), 0.0)):
        fs.reset()
        assert sum(len(f) for f in fs.process(y)) <= 1


@pytest.mark.parametrize("differential,esn0", [(True, 6.0), (False, 3.0)])
def test_sync_viterbi_rs_recovers_payloads(differential, esn0):
    """AWGN with a random carrier phase per channel (a multiple of 90 degrees in coherent mode): the synchronizer finds
    the frames and the windows decode through Viterbi and RS(64, 48) to the payloads"""
    rng = np.random.default_rng(3 + differential)
    code = R.Code(16, 48, 1)
    Cn = 24
    pays = rng.integers(0, 256, (Cn, 48)).astype(np.uint8)
    rows = []
    for c in range(Cn):
        y, pos, _ = stream(rng, b"START", [code.encode(pays[c]).tobytes()], b"END", [int(rng.integers(100, 400)), 40],
                           differential, c % 4)
        if differential:
            y = (y * np.exp(1j * rng.uniform(0, 2 * np.pi))).astype(np.complex64)
        rows.append(awgn(rng, y, esn0))
    Y = np.zeros((Cn, max(r.size for r in rows)), np.complex64)
    for c, r in enumerate(rows):
        Y[c, : r.size] = r
    fs = S.FrameSync(Cn, differential, b"START", 64, 3)
    found = fs.process(Y)
    ok = 0
    for c in range(Cn):
        if not found[c]:
            continue
        w, info = found[c][0]
        bits = V.Viterbi(1, differential).flush(w[None], w.size)[0]
        cw = np.packbits(bits[fs.P: fs.P + 8 * 64])
        msg, st = code.decode(cw)
        ok += bool(st[0] >= 0 and np.array_equal(msg, pays[c]))
    assert ok >= Cn - 1, ok
