"""CPU: the two restatements of the feed-forward AGC (tests/agc_oracle.py) agree bit for bit under any chunking, a
2^k scaling of the input changes no output bit, and behind the AGC a near-far version of the off-grid DDC scene decodes
the same frames at every level where the demodulator alone does not.  No GPU."""
import numpy as np
import pytest

from agc_oracle import AgcBatch, AgcDemod, AgcScalar, check_params
from ddc_oracle import SCENE_D, SCENE_FREQS, SCENE_FS, SCENE_RS, TSC, DdcPoly, ddc_scene, scene_taps


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _wild(rng, C, n):
    """Complex64 rows spanning 1e-30 .. 1e30 in level, with zeros, subnormals, infinities and NaNs sprinkled in."""
    x = (rng.standard_normal((C, n)) + 1j * rng.standard_normal((C, n))) * 10.0 ** rng.uniform(-30, 30, (C, n))
    x = x.astype(np.complex64)
    flat = x.reshape(-1)
    k = flat.size
    for v in (0, 1e-42 + 0j, complex(np.inf, 1), complex(1, -np.inf), complex(np.nan, 0), complex(np.nan, np.nan)):
        flat[rng.integers(0, k, max(1, k // 50))] = v
    return x


@pytest.mark.parametrize("W", [1, 2, 3, 31, 32, 33, 64, 100])
def test_scalar_and_batch_agree_bit_for_bit(W):
    rng = np.random.default_rng(W)
    x = _wild(rng, 3, 3 * W + 41)
    s, b = AgcScalar(W, 0.7, 1e6, 3), AgcBatch(W, 0.7, 1e6, 3)
    for a, c in ((0, 5), (5, 5), (5, 3 * W + 41)):                 # the second call is empty
        ys, yb = s.process(x[:, a:c]), b.process(x[:, a:c])
        assert np.array_equal(_bits(ys), _bits(yb))
    assert np.array_equal(_bits(s.gain), _bits(b.gain))


@pytest.mark.parametrize("W", [1, 2, 31, 64, 1000, 4096])
def test_any_chunking_gives_the_same_bits(W):
    rng = np.random.default_rng(100 + W)
    n = 3 * W + 500
    x = _wild(rng, 4, n)
    want = AgcBatch(W, 1.0, 1e4, 4).process(x)
    agc = AgcBatch(W, 1.0, 1e4, 4)
    parts, a = [], 0
    while a < n:
        c = min(int(rng.choice([0, 1, W - 1, W, W + 1, int(rng.integers(0, 2 * W + 3))])), n - a)
        parts.append(agc.process(x[:, a:a + c]))
        a += c
    assert np.array_equal(_bits(np.concatenate(parts, axis=1)), _bits(want))
    agc.reset()
    assert np.array_equal(_bits(agc.process(x)), _bits(want))


def test_output_is_the_input_delayed_by_w_minus_1_and_scaled():
    """A constant-envelope input comes out W-1 samples late at level ref; the zero history gives zeros first."""
    W = 16
    x = np.full((1, 100), 4 - 3j, np.complex64)
    y = AgcBatch(W, 0.5, 1e3, 1).process(x)
    assert np.all(y[0, : W - 1] == 0)
    assert np.all(y[0, W - 1:] == np.complex64(0.5 - 0.375j))


@pytest.mark.parametrize("W", [1, 2, 31, 64, 1000])
def test_scaling_by_a_power_of_two_changes_no_output_bit(W):
    rng = np.random.default_rng(7 * W)
    mag = 10.0 ** rng.uniform(-1, 1, (2, 4 * W + 300))                # envelope in [0.1, 10]: ref/m stays far below max_gain
    ph = np.exp(2j * np.pi * rng.uniform(0, 1, mag.shape))
    x = (mag * ph).astype(np.complex64)
    want = AgcBatch(W, 1.0, 1e6, 2).process(x)
    for k in range(-10, 7):
        xs = (x * np.float32(2.0 ** k)).astype(np.complex64)
        assert np.array_equal(_bits(xs), _bits(x * np.complex64(2.0 ** k)))
        assert np.array_equal(_bits(AgcBatch(W, 1.0, 1e6, 2).process(xs)), _bits(want)), k


def test_parameter_checks():
    with pytest.raises(NotImplementedError):
        check_params(0, 1.0, 1.0)
    with pytest.raises(NotImplementedError):
        check_params(4097, 1.0, 1.0)
    for ref, mg in ((0.0, 1.0), (-1.0, 1.0), (np.inf, 1.0), (np.nan, 1.0), (1.0, 0.0), (1.0, np.inf), (1.0, np.nan)):
        with pytest.raises(ValueError):
            check_params(1, ref, mg)


# ---- near-far scene ------------------------------------------------------------------------------------------------
SCENE_W = 64                                  # the AGC window of the scene: 16 symbols at 4 samples per symbol
SCENE_OFFSET = 0.001                          # residual carrier offset, cycles per sample at the channel rate
LEVELS = [2.0 ** k for k in range(-7, 4)]
# frames decoded of six without the stage, per level: the loops' gains scale with amplitude
DECODED_WITHOUT_AGC = [0, 0, 0, 0, 0, 0, 4, 5, 6, 6, 6]


def scene_rows(orc, level, seed=5):
    """The off-grid DDC scene through DdcPoly, each row scaled by `level`, given the residual offset and SCENE_W-1 zeros
    at the end (what the AGC holds back); complex64 [6, n] and the payloads."""
    h = scene_taps()
    wide, pays = ddc_scene(orc, h, SCENE_D, SCENE_FREQS, seed=seed)
    y = DdcPoly(h, SCENE_FREQS, SCENE_D).process(wide)
    rot = np.exp(2j * np.pi * SCENE_OFFSET * np.arange(y.shape[1]))
    rows = np.concatenate([y * level * rot, np.zeros((y.shape[0], SCENE_W - 1))], axis=1)
    return rows.astype(np.complex64), pays


@pytest.mark.parametrize("use_fll", [False, True])
def test_near_far_scene_decodes_at_every_level_with_the_stage(orc, use_fll):
    decoded_plain, decoded_agc = [], []
    for level in LEVELS:
        rows, pays = scene_rows(orc, level)
        plain = AgcDemod(orc, SCENE_FS, SCENE_RS, 0.35, 10, channels=len(pays), tsc=TSC, use_fll=use_fll)
        agc = AgcDemod(orc, SCENE_FS, SCENE_RS, 0.35, 10, channels=len(pays), tsc=TSC, use_fll=use_fll)
        agc.set_agc(SCENE_W, 1.0, 65536.0)
        decoded_plain.append(sum(g == p for g, p in zip(plain.DeModulateBytes(rows, b"START", b"END"), pays)))
        decoded_agc.append(sum(g == p for g, p in zip(agc.DeModulateBytes(rows, b"START", b"END"), pays)))
    assert decoded_agc == [6] * len(LEVELS)
    assert decoded_plain == DECODED_WITHOUT_AGC


def test_near_far_rows_in_one_batch(orc):
    """Six carriers, one batch, levels 2^-7 .. 2^3 spread over the rows: every frame decodes behind the AGC."""
    rows, pays = scene_rows(orc, 1.0)
    lv = np.float32(2.0) ** np.array([-7, -5, -3, -1, 1, 3], np.float32)
    rows = (rows * lv[:, None]).astype(np.complex64)
    agc = AgcDemod(orc, SCENE_FS, SCENE_RS, 0.35, 10, channels=len(pays), tsc=TSC)
    agc.set_agc(SCENE_W, 1.0, 65536.0)
    assert agc.DeModulateBytes(rows, b"START", b"END") == pays
