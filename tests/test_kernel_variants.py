"""CPU checks of the dispatch restatements in tests/kernel_variants.py: over public inputs that cross every threshold, the
FLL, modulator, equalizer and channelizer launchers reach exactly the instantiations compiled into the library, and the row
tables the GPU parity tests run cover all of them; spot values at each threshold; the FLL's create-time size limit."""
import ctypes as C_
import itertools

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


def test_names_normalise_to_one_form():
    n = kv.normalise
    assert n("void qpsk::<unnamed>::fll_duo_kernel<(int)5, (int)0, (int)4>(qpsk::FllParams, const float *)") == "fll_duo_kernel<5, 0, 4>"
    assert n("void qpsk::(anonymous namespace)::fll_duo_kernel<5, 0, 4>(qpsk::FllParams, float const*)") == "fll_duo_kernel<5, 0, 4>"
    assert n("void qpsk::mod_shape_kernel<(int)24, (int)8>(qpsk::ModArgs)") == n("void qpsk::mod_shape_kernel<24, 8>(qpsk::ModArgs)")
    assert n("qpsk::fll_group_kernel(qpsk::FllParams, const float *)") == "fll_group_kernel"
    assert n("void qpsk::pfb_history_kernel(const float2 *)") is None
    assert n("void qpsk::mod_tile_rot_kernel(qpsk::ModArgs)") is None


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
