"""CPU checks of the symbol-stage dispatch restatement (tests/symsync_dispatch.py): the geometry table has the tap counts
its rows claim, and the rows the GPU tests run reach every symsync_decode_kernel variant the dispatch can produce — every
(DIFF, MFW, DENSE, taps path, ring size) that some public input selects — while every combination no input selects is
named unreachable, with its reason."""
import itertools
import re

import symsync_dispatch as sd

SM = 148                                   # B200; the DENSE threshold scales with the SM count, the set of variants does not
DENSE_C = 96 * SM + 33
MATRIX_C = 33


def _key(v):
    return (v["diff"], v["mfw"], v["dense"], v["taps"], v["ring"])


def test_geometry_rows_have_their_tap_counts():
    for name, (fs, rs, span) in sd.GEOMETRIES.items():
        n = sd.n_taps(fs, rs, span)
        assert n == int(re.match(r"\d+", str(name)).group()), (name, n)       # a row is named by its tap count
    # the reference's banker's rounding of the rate: 2.5 -> 2, 1.25 -> 1
    assert sd.n_taps(5000, 2000, 10) == 21 and sd.n_taps(5000, 4000, 10) == 11


def test_prediction_spot_values():
    p = sd.predict
    assert p(1, 4000, 1000, 10)["mfw"] == 0                      # one stream keeps the separate filter
    assert p(31, 4000, 1000, 10)["mfw"] == 0 and p(32, 4000, 1000, 10)["mfw"] == 4
    assert p(33, 2000, 1000, 14)["mfw"] == 2 and p(33, 2000, 1000, 15)["mfw"] == 4          # 29 / 31 taps at sps 2
    assert p(33, 8000, 1000, 10)["mfw"] == 0                     # 81 taps
    assert p(33, 4000, 1000, 10, exact=False)["mfw"] == 0        # FAST matched filter: never fused
    assert p(33, 5500, 5000, 10) is None                         # sps - 0.1 <= 1: no symbol-stage kernel at all
    assert not p(96 * SM, 2000, 1000, 10, sm_count=SM)["dense"]  # grid of exactly 3 x SM
    assert p(96 * SM + 1, 2000, 1000, 10, sm_count=SM)["dense"]
    assert not p(96 * SM + 33, 4000, 1000, 10, sm_count=SM)["dense"]                       # four filter warps
    assert p(33, 2000, 1000, 16)["ring"] == 96 and p(33, 3000, 1000, 11)["ring"] == 128   # 33 / 34 taps
    assert p(33, 2000, 1000, 3)["taps"] == "const_short" and p(33, 2000, 1000, 15)["taps"] == "reg3"
    assert sd.kernel_name(p(33, 2000, 1000, 12, diff=False)) == "symsync_decode_kernel<false, 2, false>"


def _reachable():
    """Every variant a public input selects: rates (integer 2..70 and non-integer ones down to the lowest fused rate),
    spans 0..70, channel counts on both sides of the fusion and DENSE thresholds, both filter modes, both DIFF."""
    rates = [(1000 * k, 1000) for k in range(2, 71)] + [(5000, 2000), (5000, 4000), (3700, 1000), (2300, 2000), (1150, 1000)]
    out = set()
    for (fs, rs), span, C, exact, diff in itertools.product(rates, range(71), (1, 31, 32, 33, 96 * SM, DENSE_C),
                                                           (True, False), (True, False)):
        v = sd.predict(C, fs, rs, span, diff=diff, exact=exact, sm_count=SM)
        if v is not None:
            out.add(_key(v))
    return out


def _covered():
    out = set()
    for diff in (True, False):
        for row in sd.MATRIX_ROWS:
            out.add(_key(sd.predict(MATRIX_C, *sd.GEOMETRIES[row], diff=diff, sm_count=SM)))
        for row in sd.DENSE_ROWS:
            out.add(_key(sd.predict(DENSE_C, *sd.GEOMETRIES[row], diff=diff, sm_count=SM)))
            out.add(_key(sd.predict(96 * SM, *sd.GEOMETRIES[row], diff=diff, sm_count=SM)))
    return out


def test_geometry_table_reaches_every_variant_the_dispatch_can_produce():
    reachable, covered = _reachable(), _covered()
    assert reachable - covered == set(), sorted(reachable - covered, key=str)
    assert covered <= reachable
    full = itertools.product((True, False), (0, 2, 4), (False, True), sd.TAPS_CLASSES + (None,), (96, 128, None))
    for diff, mfw, dense, taps, ring in full:
        why = sd.unreachable_reason(mfw, dense, taps, ring)
        if (diff, mfw, dense, taps, ring) in reachable:
            assert why is None, ((diff, mfw, dense, taps, ring), why)
        else:
            assert why is not None, ("neither reached nor explained", (diff, mfw, dense, taps, ring))
    # DIFF x {MFW 0, 2, 2-DENSE, 4} x {NB 1, 2, 3, constant bank short, long} x {ring 96, 128}: 19 variants per DIFF
    assert len(reachable) == 2 * 19, len(reachable)


def test_chunk_spot_values():
    assert sd.chunks(2047, 256, True) == 1 and sd.chunks(2048, 256, True) == 6        # the pipeline starts at 2048 samples
    assert sd.chunks(4196, 4096, True) == 6 and sd.chunks(4196, 4097, True) == 4
    assert sd.chunks(4196, 256, False) == 1                                           # device source, no FLL: one launch
    assert sd.chunks(4196, 1024, False, host=True) == 4 and sd.chunks(4196, 1024, False, host=True, cs16=True) == 2
    assert sd.chunks(4196, 16384, False, host=True) == 6                              # at most six copy chunks
    assert sd.chunks(300, 16384, False, host=True) == 1                               # chunks of >= 256 samples
    assert sd.chunks(4196, 2048, True, host=True, fused=False) == 1                   # unfused calls: one chunk


def test_route_rows_reach_every_route():
    got = {name: sd.route(row) for name, row in sd.ROUTE_ROWS.items()}
    assert {r for r, _ in got.values()} == set(sd.ROUTES), got
    assert {n for _, n in got.values()} >= {1, 2, 4, 6}, got
    assert all(n == 1 for r, n in got.values() if not r.startswith("pipeline")), got
