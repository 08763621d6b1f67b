"""CPU checks of tests/bank_bounds.py: the fp64 references equal the polyphase restatements of the oracles, the row tables
have the shapes the GPU test needs, and on every row each tap, history, phase and index slip moves the reference by more
than ten times the per-output bound, so that a kernel making that slip could not pass tests/test_gpu_bank_bounds.py."""
import numpy as np
import pytest

import bank_bounds as bb
import kernel_variants as kv
from ddc_oracle import DdcPoly
from pfb_oracle import PfbPoly
from resamp_oracle import ResampPoly, resamp_count

CASES = [(block, row) for block in ("resamp", "ddc", "pfb") for row in bb.block_rows(block)]


def _oracle(block, row, h, xs):
    if block == "resamp":
        o = ResampPoly(h, row[1], row[2], row[0])
    elif block == "ddc":
        o = DdcPoly(h, bb.ddc_freqs(row[0]), row[1])
    else:
        o = PfbPoly(h, row[1])
    return [o.process(x) for x in xs]


@pytest.mark.parametrize("block,row", CASES, ids=[bb.row_id(b, r) for b, r in CASES])
def test_bound_sees_every_slip(block, row):
    h, xs, ref, mutations = bb.row_case(block, row)
    assert np.all(h != 0) and (row[-1] == "kaiser" or h.size < 2 or h[-1] * h[-2] < 0)
    base = ref(h, xs)
    for k, ((y, br, bi), want) in enumerate(zip(base, _oracle(block, row, h.astype(np.float64), xs))):
        assert y.shape == want.shape and y.shape[1] > 0, (k, y.shape, want.shape)
        assert np.abs(y - want).max() <= 1e-12 * np.abs(want).max(), k
    moved = {}
    for mu in mutations:
        moved[mu] = 0.0
        for (y, br, bi), (my, _, _) in zip(base, ref(h, xs, mu)):
            d = my - y
            moved[mu] = max(moved[mu], float((np.abs(d.real) / br).max()), float((np.abs(d.imag) / bi).max()))
    hidden = {mu: f"{moved[mu]:.3g}" for mu in bb.promised(block, row, mutations) if not moved[mu] > 10.0}
    assert not hidden, ("slips within ten times the bound", hidden)


def test_every_mutation_is_run_on_the_random_tap_rows():
    for block, muts, of in (("resamp", bb.RESAMP_MUTATIONS, bb.resamp_mutations), ("ddc", bb.DDC_MUTATIONS, bb.ddc_mutations),
                            ("pfb", bb.PFB_MUTATIONS, bb.pfb_mutations)):
        run = set().union(*(of(row) for row in bb.block_rows(block) if row[-1] == "rand"))
        assert run == set(muts), (block, set(muts) - run)
    assert {"q = P-1 dropped in branch M-1", "twiddle conjugated"} <= set(bb.pfb_mutations((16, 1024, "kaiser")))


def test_rows_have_the_shapes_the_gpu_test_needs():
    # resampler: both shapes at K = 8 | 9; L > M, L < M, L = 1; P = 1 and 64; several tiles per call, ragged
    rs = kv.RESAMP_ROWS
    assert {K for K, *_ in rs} == {8, 9}
    assert any(L > M for _, L, M, _, _ in rs) and any(L < M for _, L, M, _, _ in rs) and any(L == 1 for _, L, _, _, _ in rs)
    assert {-(-N // L) for _, L, _, N, _ in rs} >= {1, 64}
    for K, L, M, N, kind in rs:
        a = 0
        for n in kv.resamp_row_calls((K, L, M)):
            t = resamp_count(a + n, L, M) - resamp_count(a, L, M)
            tile = kv.RESAMP_TILE[K <= kv.RESAMP_SMALL_K]
            assert t > 3 * tile and t % tile, (K, L, M, t)
            a += n
    # DDC: both shapes; several tiles, ragged; pending samples at the seam wherever D > 1
    for K, D, N, kind in kv.DDC_ROWS:
        n1, n2 = kv.ddc_row_calls((K, D))
        tile = kv.DDC_TILE[K <= kv.DDC_SMALL_K]
        for t in (n1 // D, (n1 + n2) // D - n1 // D):
            assert t > 3 * tile and t % tile
        assert D == 1 or n1 % D
    assert {K for K, *_ in kv.DDC_ROWS} == {8, 9} and {D for _, D, _, _ in kv.DDC_ROWS} >= {1, 16, 64}
    # channelizer: every channelizer row, every P at M = 4 and 1024, several tiles and a pending sample at the seam
    assert [(P, M) for P, M, kind in bb.PFB_BANK_ROWS if kind == "rand"] == kv.PFB_ROWS
    for row in bb.PFB_BANK_ROWS:
        P, M, _ = row
        n1, n2 = bb.pfb_row_calls(row)
        assert n1 // M > 3 * (bb.PFB_TILE_BLOCKS // M) and n1 % M
    # one Kaiser row per block
    assert sum(r[-1] == "kaiser" for r in kv.DDC_ROWS) == 2 and sum(r[-1] == "kaiser" for r in kv.RESAMP_ROWS) == 2
    assert sum(r[-1] == "kaiser" for r in bb.PFB_BANK_ROWS) == 1


def test_inputs_span_the_levels_the_bounds_must_see():
    xs = bb.resamp_row_inputs((9, 5, 8, 120, "rand"))
    peak = np.abs(np.concatenate(xs, axis=1)).max(axis=1)
    assert peak[0] < 2.0 ** -19 and peak[-1] > 2.0 ** 19                # batch rows 2^-20 .. 2^20
    K = 9
    y = bb.ddc_reference(bb.ddc_row_taps((K, 16, 128, "kaiser")), bb.ddc_freqs(K), 16,
                         bb.ddc_row_inputs((K, 16, 128, "kaiser")))[0][0]
    lvl = np.median(np.abs(y), axis=1)
    assert lvl[1] < 2e-3 * np.abs(y[0]).max()      # the -60 dB carrier's channel: below what 1e-5 max|y| can judge
    assert min(abs(f) for f in bb.ddc_freqs(K)) > 0.05


def test_kaiser_prototype_is_the_librarys(qp):
    h = qp.pfb_taps(1024, 16, 0.5 / 1024, 60.0)
    assert np.abs(bb.kaiser_pfb(1024, 16) - h).max() <= 1e-12 * np.abs(h).max()


def test_pfb_dif_is_the_inverse_dft():
    rng = np.random.default_rng(3)
    for M in (2, 4, 8, 64, 1024):
        v = rng.standard_normal((3, M)) + 1j * rng.standard_normal((3, M))
        want = np.fft.ifft(v, axis=1) * M
        assert np.abs(bb.pfb_dif(v, bb.pfb_twiddles(M)) - want).max() <= 1e-10 * np.abs(want).max()
