"""CPU checks of the dispatch restatements in tests/kernel_variants.py: over public inputs that cross every threshold, the
FLL, modulator, equalizer, channelizer and FIR launchers reach exactly the instantiations compiled into the library, and the
row tables the GPU parity tests run cover all of them; spot values at each threshold; every tap-loop tail of the FIR kernels
in the FIR table, and a bound that sees a dropped or misplaced tap on every FIR row; the FLL's create-time size limit."""
import ctypes as C_
import itertools

import numpy as np
import pytest

import kernel_variants as kv


@pytest.fixture(scope="module")
def built(qp):
    return kv.compiled(qp._native.LIB_PATH)


def _reachable(family):
    out = set()
    if family == "fll":
        sizes = list(range(1, 80)) + [286, 287, 1000, 1430, 1431, 2048]
        for n, c in itertools.product(sizes, (1, 5, 1280, 1281, 5119, 5120, 16384)):
            for phase, sps in ((0.0, 4.0), (31.0, 4.0), (32.0, 4.0), (2e4, 4.0), (0.0, 1e-4)):
                out.add(kv.fll_predict(n, c, phase=phase, sps=sps))
    elif family == "mod":
        rates = [(1000 * s, 1000) for s in range(1, 20)] + [(2500, 1000), (5000, 2000), (256000, 1000), (257000, 1000),
                                                            (3500, 1000), (1500, 1000)]
        for (fs, rs), span, pulse in itertools.product(rates, range(0, 200), (True, False)):
            out.add(kv.mod_predict(fs, rs, span, pulse))
    elif family == "eq":
        for n, sps in itertools.product(range(0, 70), range(0, 10)):
            out.add(kv.eq_predict(n, sps))
    elif family == "pfb":
        for M, n in itertools.product((1, 2, 3, 4, 8, 64, 256, 1024, 2048), range(1, 40 * 64)):
            out.add(kv.pfb_predict(n, M))
        for n in range(1, 34 * 1024, 97):
            out.add(kv.pfb_predict(n, 1024))
    elif family == "ddc":
        for n, c, d in itertools.product((0, 1, 100, 4096, 4097), list(range(0, 40)) + [2047, 2048, 2049], (0, 1, 1024, 1025)):
            out.add(kv.ddc_predict(n, c, d))
    elif family == "resamp":
        for n, L, M, c in itertools.product((0, 1, 64, 65, 16384, 16385), (0, 1, 256, 1024, 1025), (0, 1, 1024, 1025),
                                            list(range(0, 40)) + [16383, 16384, 16385]):
            out.add(kv.resamp_predict(n, L, M, c))
    elif family == "fir":
        sizes = sorted(set(range(1, 140)) | set(range(140, 1100, 13)) |
                       {n + d for n in (256, 512, 536, 560, 600, 889, 1039) for d in (-1, 0, 1, 2)})
        L = 5000
        layouts = [(0, 0, 1, L, L), (1, 0, 1, L, L), (0, 1, 1, L, L), (0, 0, 3, L + 1, L), (0, 0, 3, L, L + 1),
                   (0, 0, 3, L + 2, L + 2)]
        for n, cplx, mode, (xo, yo, C, ldx, ldy) in itertools.product(sizes, (False, True), kv.FIR_MODES, layouts):
            for op, skip in (("filter", 0), ("fft", 0), (1, 0), (3, 2), (2, 0), (2, 1), (4, 3), (8, 6), (16, 5)):
                out.update(kv.fir_predict(n, cplx, mode, op, L, skip, xo, yo, C, ldx, ldy))
    out.discard(kv.UNSUPPORTED)
    return out


def _covered(family):
    return set(kv.predicted_launches(family)) - {kv.UNSUPPORTED}


@pytest.mark.parametrize("family", sorted(kv.FAMILIES))
def test_dispatch_reaches_exactly_the_compiled_instantiations(built, family):
    reachable, compiled = _reachable(family), built[family]
    assert compiled, f"no {family} kernel found in the library"
    assert not compiled - reachable, ("compiled but reached by no input", sorted(compiled - reachable))
    assert not reachable - compiled, ("predicted but not compiled", sorted(reachable - compiled))


@pytest.mark.parametrize("family", sorted(kv.FAMILIES))
def test_row_tables_cover_every_reachable_instantiation(family):
    reachable, covered = _reachable(family), _covered(family)
    assert not reachable - covered, ("no table row reaches", sorted(reachable - covered))
    assert covered <= reachable
    assert kv.UNSUPPORTED not in kv.predicted_launches(family)


def test_instantiation_counts():
    assert len(_reachable("fll")) == 96 + 2 + 1           # fll_duo_kernel<K, TAIL, PAIRS>, fll_pair_kernel<10 / 40>, generic
    assert len(_reachable("mod")) == 52
    assert len(_reachable("eq")) == 40
    assert len(_reachable("pfb")) == 32
    assert len(_reachable("ddc")) == 2                    # ddc_kernel<1, 1, 8> for K <= 8, <4, 2, 32> above
    assert len(_reachable("resamp")) == 2                 # resamp_kernel<1, 1, 1, 2048> for K <= 8, <32, 2, 4, 64> above
    assert len(_reachable("fir")) == 3 + 1 + 1 + 2 + 1 + 3 + 4 + 1    # ... + fir_decim_kernel<D = 2..16>, fir_subsample_kernel


def test_names_normalise_to_one_form():
    n = kv.normalise
    assert n("void qpsk::<unnamed>::fll_duo_kernel<(int)5, (int)0, (int)4>(qpsk::FllParams, const float *)") == "fll_duo_kernel<5, 0, 4>"
    assert n("void qpsk::(anonymous namespace)::fll_duo_kernel<5, 0, 4>(qpsk::FllParams, float const*)") == "fll_duo_kernel<5, 0, 4>"
    assert n("void qpsk::mod_shape_kernel<(int)24, (int)8>(qpsk::ModArgs)") == n("void qpsk::mod_shape_kernel<24, 8>(qpsk::ModArgs)")
    assert n("qpsk::fll_group_kernel(qpsk::FllParams, const float *)") == "fll_group_kernel"
    assert n("void qpsk::pfb_history_kernel(const float2 *)") is None
    assert n("void qpsk::mod_tile_rot_kernel(qpsk::ModArgs)") is None
    assert n("void qpsk::fir_tma_kernel<(int)10, (int)256, (bool)0>(qpsk::FirArgs, qpsk::TapsReal)") == "fir_tma_kernel<10, 256, false>"
    assert n("void qpsk::fir_tma_kernel<10, 256, false>(qpsk::FirArgs, qpsk::TapsReal)") == "fir_tma_kernel<10, 256, false>"
    assert n("void qpsk::fir_decim_tma_kernel<(int)7, (int)64, (int)4, (int)8, (bool)1>(qpsk::FirArgs, qpsk::TapsReal)") == \
        n("void qpsk::fir_decim_tma_kernel<7, 64, 4, 8, true>(qpsk::FirArgs const, qpsk::TapsReal const)") == \
        "fir_decim_tma_kernel<7, 64, 4, 8, true>"
    assert n("void qpsk::fir_decim_kernel<(int)7, (int)256, (int)1, (int)2>(qpsk::DecArgs, qpsk::TapsReal)") == \
        "fir_decim_kernel<7, 256, 1, 2>"
    assert n("qpsk::fir_subsample_kernel(const float2 *, long long, long long, int, long long, float2 *, long long, int)") == \
        "fir_subsample_kernel"
    assert n("void qpsk::fir_hist_update_kernel(const float2 *, long long, long long, const float2 *, float2 *, int, int)") is None


def test_fll_spot_values():
    p = kv.fll_predict
    assert p(40, 1280) == "fll_duo_kernel<5, 0, 1>" and p(40, 1281) == "fll_duo_kernel<5, 0, 4>"
    assert p(40, 5119) == "fll_duo_kernel<5, 0, 4>" and p(40, 5120) == "fll_pair_kernel<40>"
    assert p(10, 5120) == "fll_pair_kernel<10>" and p(13, 5120) == "fll_duo_kernel<1, 5, 4>"
    assert p(40, 5120, phase=32.0) == "fll_duo_kernel<5, 0, 4>"        # far phase: the two-warp kernel for one call
    assert p(40, 5120, phase=2e4) == "fll_group_kernel"                # wild state
    assert p(40, 5, sps=1e-4) == "fll_group_kernel"                    # frequency limit beyond the short-range sin/cos
    assert p(7, 5) == "fll_group_kernel" and p(8, 5) == "fll_duo_kernel<1, 0, 1>"
    assert p(55, 5) == "fll_duo_kernel<6, 7, 1>" and p(56, 5) == "fll_group_kernel"
    # 48 / 49 taps: the two-warp kernel's ring grows from 64 to 128 slots (N + 16 <= 64)
    assert p(48, 5) == "fll_duo_kernel<6, 0, 1>" and p(49, 5) == "fll_duo_kernel<6, 1, 1>"
    assert 48 + 16 <= 64 < 49 + 16
    # the generic kernel's shared memory: 48 KiB up to 286 taps (287 needs the opt-in), 200 KiB up to 1430
    assert kv.fll_group_smem(286) <= 48 * 1024 < kv.fll_group_smem(287)
    assert kv.fll_max_size() == 1430
    assert p(1430, 1) == "fll_group_kernel" and p(1431, 1) == kv.UNSUPPORTED and p(2048, 1) == kv.UNSUPPORTED


def test_modulator_spot_values():
    p = kv.mod_predict
    for sps in (2, 4, 8):                                             # m 24 -> 32: the compile-time rate ends at MT 24
        assert p(1000 * sps, 1000, 23) == f"mod_shape_kernel<24, {sps}>"
        assert p(1000 * sps, 1000, 24) == "mod_shape_kernel<32, 0>"
    assert p(2000, 1000, 95) == "mod_shape_kernel<96, 0>"             # m = 96
    assert p(2000, 1000, 96) == kv.UNSUPPORTED                        # m = 97
    assert p(2000, 1000, 96, pulse=False) == "mod_shape_kernel<64, 0>"   # the delta bank: delay + 1 = 97 taps, m = 49
    assert p(256000, 1000, 4) == "mod_shape_kernel<5, 0>" and p(256000, 1000, 4, pulse=False) == "mod_shape_kernel<4, 0>"
    assert p(257000, 1000, 4) == kv.UNSUPPORTED and p(257000, 1000, 4, pulse=False) == kv.UNSUPPORTED
    assert p(3000, 1000, 10) == "mod_shape_kernel<11, 0>" and p(4000, 1000, 10) == "mod_shape_kernel<11, 4>"
    assert p(2500, 1000, 6) == "mod_shape_kernel<7, 2>"               # 2.5 rounds to 2 taps per symbol, sps 2: 13 taps
    assert kv.mod_taps(2500, 1000, 6) == 13 and kv.mod_taps(3500, 1000, 2) == 9   # banker's rounding: 2.5 -> 2, 3.5 -> 4
    assert p(4000, 1000, 0) == "mod_shape_kernel<4, 4>"               # one tap


def test_equalizer_spot_values():
    p = kv.eq_predict
    assert p(8, 1) == "cma_eq_kernel<1, 1>" and p(9, 1) == "cma_eq_kernel<2, 1>"
    assert p(56, 2) == "cma_eq_kernel<7, 2>" and p(57, 2) == "cma_eq_kernel<8, 2>" and p(64, 8) == "cma_eq_kernel<8, 8>"
    for sps in (3, 5, 6, 7):
        assert p(21, sps) == "cma_eq_kernel<3, 0>"
    assert p(65, 1) == kv.UNSUPPORTED and p(21, 9) == kv.UNSUPPORTED and p(0, 1) == kv.UNSUPPORTED


def test_channelizer_spot_values():
    p = kv.pfb_predict
    assert p(4, 4) == "pfb_kernel<1>" and p(5, 4) == "pfb_kernel<2>" and p(32 * 1024, 1024) == "pfb_kernel<32>"
    assert p(32 * 1024 + 1, 1024) == kv.UNSUPPORTED and p(16, 6) == kv.UNSUPPORTED
    assert all(p(kv.pfb_taps(P, M), M) == f"pfb_kernel<{P}>" for P in range(1, 33) for M in (4, 1024))


def test_ddc_and_resampler_spot_values():
    d, r = kv.ddc_predict, kv.resamp_predict
    assert d(128, 8, 16) == "ddc_kernel<1, 1, 8>" and d(128, 9, 16) == "ddc_kernel<4, 2, 32>"
    assert d(4096, 2048, 1024) == "ddc_kernel<4, 2, 32>" and d(1, 1, 1) == "ddc_kernel<1, 1, 8>"
    assert d(4097, 8, 16) == d(128, 2049, 16) == d(128, 8, 1025) == d(0, 8, 16) == kv.UNSUPPORTED
    assert r(3000, 125, 128, 8) == "resamp_kernel<1, 1, 1, 2048>" and r(3000, 125, 128, 9) == "resamp_kernel<32, 2, 4, 64>"
    assert r(64, 1, 1, 16384) == "resamp_kernel<32, 2, 4, 64>" and r(65, 1, 1, 1) == kv.UNSUPPORTED    # P = 65
    assert r(16384, 256, 1, 1) == "resamp_kernel<1, 1, 1, 2048>" and r(16385, 1024, 1, 1) == kv.UNSUPPORTED
    assert r(8, 1025, 1, 1) == r(8, 1, 1025, 1) == r(8, 1, 1, 16385) == r(0, 1, 1, 1) == kv.UNSUPPORTED


def test_fir_spot_values():
    p = kv.fir_predict
    tma, tma_w, tma_c = "fir_tma_kernel<10, 256, false>", "fir_tma_kernel<10, 320, false>", "fir_tma_kernel<10, 256, true>"
    split, exact, gen, gen_x = ("fir_split2_kernel<10, 256>", "fir_exact_real_kernel<256>", "fir_generic_kernel<false>",
                                "fir_generic_kernel<true>")
    # FAST: the split kernel from G = 48 (45 / 46 streaming taps), SPLIT mode from G = 14
    assert p(45) == [tma] and p(46) == [split] and p(11, mode="SPLIT") == [tma] and p(12, mode="SPLIT") == [split]
    # FMA: ten consumer warps for real taps at G = 48..96 (46..95 streaming taps, 47..96 stateless; EXACT is FMA when stateless)
    assert p(45, mode="FMA") == [tma] and p(46, mode="FMA") == [tma_w] and p(95, mode="FMA") == [tma_w]
    assert p(96, mode="FMA") == [tma] and p(46, True, "FMA") == [tma_c]
    for mode in ("FMA", "EXACT"):
        assert p(46, mode=mode, op="fft") == [tma] and p(47, mode=mode, op="fft") == [tma_w]
        assert p(96, mode=mode, op="fft") == [tma_w] and p(97, mode=mode, op="fft") == [tma]
    # the split kernel's ring fits up to 889 streaming taps
    assert p(889) == [split] and p(890) == [tma]
    # EXACT: the exact-order TMA kernel from 8 to 513 taps (HL = 512, a whole tile of halo); odd strides and offsets leave it
    assert p(7, mode="EXACT") == [gen_x] and p(8, mode="EXACT") == [exact]
    assert p(513, mode="EXACT") == [exact] and p(514, mode="EXACT") == [gen_x]
    assert p(64, mode="EXACT", x_off=1) == [gen_x] and p(64, mode="EXACT", channels=3, ldx=1001, ldy=1000) == [gen_x]
    assert p(21, True, "EXACT") == [gen_x]
    # kMaxG = 1040: 1039 / 1040 streaming taps, 1040 / 1041 stateless
    for cplx, k in ((False, tma), (True, tma_c)):
        assert p(1039, cplx, "FMA") == [k] and p(1040, cplx, "FMA") == [gen]
        assert p(1040, cplx, "FMA", "fft") == [k] and p(1041, cplx, "FMA", "fft") == [gen]
    assert p(1039) == [tma] and p(1040) == [gen]
    # decimators: the TMA ring at D = 8 / 16 fits up to 535 / 559 taps, then the register-staged kernel
    assert kv.fir_decim_tma_limit(8) == 535 and kv.fir_decim_tma_limit(16) == 559 and kv.fir_decim_tma_limit(4) == 1039
    assert p(535, op=8) == ["fir_decim_tma_kernel<7, 64, 4, 8, true>"] and p(536, op=8) == ["fir_decim_kernel<7, 64, 4, 8>"]
    assert p(559, op=16) == ["fir_decim_tma_kernel<7, 32, 8, 16, true>"] and p(560, op=16) == ["fir_decim_kernel<7, 32, 8, 16>"]
    # K * D > kMaxG: the full-rate filter and the subsampling kernel, for every D
    fast = {2: "fir_dec2_kernel<14, 256>", 4: "fir_decim_tma_kernel<7, 128, 2, 4, false>", 8: "fir_decim_kernel<7, 64, 4, 8>",
            16: "fir_decim_kernel<7, 32, 8, 16>"}
    for D, k in fast.items():
        assert p(1039, op=D, skip=1) == [k] and p(1040, op=D, skip=1) == [gen, "fir_subsample_kernel"]
    assert (kv.fir_hl(1039) + 1 + 1 + 1) & ~1 == kv.kMaxG                 # Gs of fir_dec2_kernel at the kept phase 1
    # layouts: offsets and odd strides leave the bulk-copy kernels; the output pointer does not matter for D >= 4
    assert p(65, op=2, x_off=1) == p(65, op=2, y_off=1) == ["fir_decim_kernel<7, 256, 1, 2>"]
    assert p(65, op=4, y_off=1) == ["fir_decim_tma_kernel<7, 128, 2, 4, false>"]
    assert p(65, op=4, x_off=1) == ["fir_decim_kernel<7, 128, 2, 4>"]
    assert p(65, op=8, channels=3, ldx=1001, ldy=1000) == ["fir_decim_kernel<7, 64, 4, 8>"]
    assert p(65, op=8, channels=3, ldx=1000, ldy=1001) == ["fir_decim_tma_kernel<7, 64, 4, 8, true>"]
    assert p(33, x_off=1) == [gen] and p(33, channels=3, ldx=1000, ldy=1001) == [gen]
    # the full-rate path: odd D, D = 1, complex taps, EXACT mode; nothing to subsample, no subsampling kernel
    assert p(129, op=3) == [split, "fir_subsample_kernel"] and p(33, op=1) == [tma, "fir_subsample_kernel"]
    assert p(40, True, op=4) == [tma_c, "fir_subsample_kernel"] and p(65, mode="EXACT", op=8) == [exact, "fir_subsample_kernel"]
    assert p(33, op=4, L=3, skip=3) == [tma]


def test_fir_table_holds_every_tail_residue():
    seen = {}
    for r in kv.FIR_ROWS:
        for call in kv.fir_row_dispatch(r):
            for k, t in call:
                seen.setdefault(k, set()).add(t)
    for k, ts in seen.items():
        base = k.split("<")[0]
        if base not in kv.FIR_TAIL_MOD:
            continue
        mod = kv.FIR_TAIL_MOD[base]
        want = set(range(0, mod, 2)) if base == "fir_tma_kernel" else set(range(mod))   # G is even
        assert ts == want, (k, sorted(want - ts))
    assert set(seen) == _reachable("fir")


def test_fir_table_has_the_shapes_the_gpu_tests_need():
    for r in kv.FIR_ROWS:
        calls = kv.fir_row_calls(r)
        assert len(calls) == 2 and calls[0]["L"] % 2 == 1, r
        if isinstance(r[3], int) and r[5]:
            assert calls[1]["skip"] == r[5] and 1 <= r[5] < r[3], r
        for c in calls:
            assert c["L"] >= 3 * 3584 + 1 and c["L"] % 3584 and c["L"] % 3200 and c["L"] % 512, r
            if r[4] == "even3":
                assert c["ldx"] % 2 == 0 and c["ldy"] % 2 == 0
                assert 3 * (c["L"] // 3584) > 2 * 148                     # more tiles than two CTAs on each of 148 SMs
            if r[4] == "odd3":
                assert c["ldx"] % 2 == 1 and c["ldy"] % 2 == 1
    assert {r[4] for r in kv.FIR_ROWS} == set(kv.FIR_LAYOUTS)
    assert {r[5] for r in kv.FIR_ROWS if r[3] == 16} >= set(range(1, 16, 2))


def _mutations(taps):
    n = taps.size // 2
    first, last = taps.copy(), taps.copy()
    first[0:2] = 0
    last[2 * n - 2:] = 0
    out = [("first tap zeroed", first), ("last tap zeroed", last)]
    if n > 1:
        swap = taps.copy()
        swap[2 * n - 4: 2 * n - 2], swap[2 * n - 2:] = taps[2 * n - 2:], taps[2 * n - 4: 2 * n - 2]
        out.append(("last two taps swapped", swap))
    return out


@pytest.mark.parametrize("row", kv.FIR_ROWS, ids=[f"{r[0]}-{r[1]}-{r[2]}-{r[3]}-{r[4]}-{r[5]}" for r in kv.FIR_ROWS])
def test_fir_bound_sees_a_dropped_or_misplaced_tap(row):
    """Each mutation moves the float64 reference by more than ten times the row's bound on some output: a kernel that
    dropped or misplaced that tap could not pass tests/test_gpu_fir_variants.py."""
    n, cplx, _, op = row[:4]
    taps = kv.fir_row_taps(row)
    assert np.all(taps[0::2] != 0) and (not cplx or np.all(taps[1::2] != 0))
    xs = kv.fir_row_inputs(row)
    refs = kv.fir_reference(taps, xs, op)
    bounds = [kv.fir_bound(call[0][0], n, cplx, ref) for call, ref in zip(kv.fir_row_dispatch(row), refs)]
    for what, t in _mutations(taps):
        moved = 0.0
        for ref, mref, (br, bi) in zip(refs, kv.fir_reference(t, xs, op), bounds):
            d = mref[0] - ref[0]
            moved = max(moved, float((np.abs(d.real) / br).max()), float((np.abs(d.imag) / bi).max()))
        assert moved > 10.0, (what, moved)


def test_row_tables_have_the_shapes_the_gpu_tests_need():
    # FLL: every two-warp size at PAIRS 1 and 4, the C = 1280 / 1281 switch, the generic kernel at 1 and 33 streams
    assert {n for n, c in kv.FLL_ROWS if c == 5} == set(range(8, 56)) == {n for n, c in kv.FLL_ROWS if c == 1300}
    assert (1300 + 15) // 16 == 82 and 1300 - 81 * 16 == 4                    # the last CTA: one live pair of four
    # equalizer: every (J, S) at 37 channels, S = 0 through sps 3 and sps 7
    assert {kv.eq_predict(n, s) for n, s in kv.EQ_ROWS} == _reachable("eq")
    assert {s for _, s in kv.EQ_ROWS if kv.eq_predict(21, s).endswith(", 0>")} == {3, 7}
    # channelizer: every P at M = 4 and at M = 1024
    for M in (4, 1024):
        assert sorted(P for P, m in kv.PFB_ROWS if m == M) == list(range(1, 33))


def test_fll_create_refuses_sizes_the_generic_kernel_cannot_run(qp):
    """1431..2048 taps were accepted at creation, and then every Process call failed.  The size check comes before the
    device is touched, so it holds on a machine without a GPU."""
    lib, N = qp._native.lib(), qp._native
    for size in (1431, 2048, 2049, 1 << 30):
        h = C_.c_void_p()
        assert lib.qpsk_fll_create(4.0, 0.35, size, 0.05, C_.byref(h)) == N.ERR_UNSUPPORTED, size
        assert lib.qpsk_fll_create_batch(4.0, 0.35, size, 0.05, 3, C_.byref(h)) == N.ERR_UNSUPPORTED, size
        assert not h.value
    h = C_.c_void_p()
    st = lib.qpsk_fll_create(4.0, 0.35, 1430, 0.05, C_.byref(h))
    assert st != N.ERR_UNSUPPORTED, st
    if h.value:
        lib.qpsk_fll_destroy(h)
