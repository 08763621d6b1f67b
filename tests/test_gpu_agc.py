"""GPU: the feed-forward AGC (csrc/agc.cu) is bit-identical to its restatement (tests/agc_oracle.py) over both kernels,
any chunking, strided and offset rows, reset and repeated runs, leaves guard bands alone and checks its arguments; the
demodulator's AGC stage is bit-identical to the oracle demodulator behind the restated AGC, keeps the fused symbol-stage
kernel (seen through the profiler), and takes the DDC bank's rows on one stream."""
import numpy as np
import pytest

from agc_oracle import AgcBatch, AgcDemod
from ddc_oracle import SCENE_D, SCENE_FREQS, SCENE_FS, SCENE_RS, TSC, ddc_scene, scene_taps
from symsync_dispatch import symsync_variants

pytestmark = pytest.mark.gpu


def _bits(a):
    """The float32 bit patterns, every NaN made the same one (a NaN's sign and payload are not specified)."""
    f = np.ascontiguousarray(a).view(np.float32).copy()
    f[np.isnan(f)] = np.float32("nan")
    return f.view(np.uint32)


def _rows(rng, C, n, spread=6.0):
    lv = 10.0 ** rng.uniform(-spread, spread, (C, 1))
    x = (rng.standard_normal((C, n)) + 1j * rng.standard_normal((C, n))) * lv * 10.0 ** rng.uniform(-1, 1, (C, n))
    x = x.astype(np.complex64)
    flat = x.reshape(-1)
    for v in (0, 1e-42 + 0j, complex(np.inf, 1), complex(np.nan, 0)):
        flat[rng.integers(0, flat.size, max(1, flat.size // 997))] = v
    return x


# tiles: W <= 32 runs floor(32/W)*W*64 outputs per warp, W > 32 W*max(8, ceil(16384/W)); the sizes span several tiles
# with a ragged end where the channel count allows
CASES = [(1, 1, 5000), (3, 2, 4500), (33, 31, 4100), (2048, 1, 300), (2048, 2, 257), (2048, 31, 150), (2048, 64, 400),
         (2048, 1000, 1100), (2048, 4096, 4200), (5, 64, 40000), (3, 1000, 40000), (2, 4096, 70000), (64, 1000, 2000),
         (17, 33, 3000), (100, 4096, 9000), (7, 32, 4097)]


@pytest.mark.parametrize("C,W,n", CASES)
def test_block_matches_restatement(gpu, C, W, n):
    rng = np.random.default_rng(C * 7919 + W * 31 + n)
    x = _rows(rng, C, n)
    want_agc = AgcBatch(W, 0.5, 1e5, C)
    want = want_agc.process(x)
    agc = gpu.Agc(W, 0.5, 1e5, C)
    got = agc.process(x)
    assert np.array_equal(_bits(got), _bits(want))
    assert np.array_equal(_bits(agc.gain), _bits(want_agc.gain))


@pytest.mark.parametrize("C,W", [(3, 1), (40, 2), (5, 31), (33, 64), (4, 1000), (2, 4096)])
def test_chunked_strided_offset_rows_reset_and_guards(gpu, C, W):
    import torch
    rng = np.random.default_rng(C + W)
    n = 3 * W + 3000
    x = _rows(rng, C, n)
    want = AgcBatch(W, 1.0, 1e4, C).process(x)
    ldx, ldy, guard = 2 * n + 6, 2 * n + 10, 8        # strides in floats: odd sample counts past the row
    xin = np.zeros((C, ldx + 2), np.float32)
    xin[:, 2:2 + 2 * n] = x.view(np.float32)                       # rows start one sample into the buffer
    agc = gpu.Agc(W, 1.0, 1e4, C)
    ts = torch.cuda.Stream()
    for rep in range(2):
        with torch.cuda.stream(ts):
            d_x_full = torch.from_numpy(xin.copy()).cuda()
            buf = torch.full((C * ldy + 2 * guard,), 7.25, dtype=torch.float32, device="cuda")
            a = 0
            while a < n:
                c = min(int(rng.choice([0, 1, W - 1, W + 1, int(rng.integers(0, 3 * W + 50))])), n - a)
                # row c starts at float 2 + c*(ldx+2) of xin: pass the row-1 start plus one sample, stride ldx+2
                agc.process_dev(d_x_full.data_ptr() + 4 * (2 + 2 * a), buf.data_ptr() + 4 * (guard + 2 * a), 2 * c,
                                ldx + 2, ldy, ts.cuda_stream)
                a += c
            ts.synchronize()
            out = buf.cpu().numpy()
        assert np.all(out[:guard] == 7.25) and np.all(out[guard + C * ldy:] == 7.25)
        rows = out[guard: guard + C * ldy].reshape(C, ldy)
        assert np.all(rows[:, 2 * n:] == 7.25)
        assert np.array_equal(_bits(np.ascontiguousarray(rows[:, : 2 * n]).view(np.complex64)), _bits(want)), rep
        agc.reset()


def test_argument_checks_and_refused_calls_consume_nothing(gpu):
    import torch
    from qpsk_modulator_demodulator_b200 import _native as N
    with pytest.raises(N.QpskCudaError):
        gpu.Agc(0)
    with pytest.raises(N.QpskCudaError):
        gpu.Agc(4097)
    for ref, mg in ((0.0, 1.0), (-1.0, 1.0), (float("inf"), 1.0), (float("nan"), 1.0), (1.0, 0.0), (1.0, float("inf"))):
        with pytest.raises(N.ArgumentOutOfRangeException):
            gpu.Agc(8, ref, mg)
    with pytest.raises(N.ArgumentOutOfRangeException):
        gpu.Agc(8, channels=0)
    rng = np.random.default_rng(3)
    C, W, n = 4, 40, 500
    x = _rows(rng, C, n)
    want = AgcBatch(W, 1.0, 65536.0, C).process(x)
    agc = gpu.Agc(W, channels=C)
    d_x = torch.from_numpy(x.view(np.float32).copy()).cuda()
    d_y = torch.zeros(C * 2 * n + 2, dtype=torch.float32, device="cuda")
    L = N.lib()
    x0, y0 = d_x.data_ptr(), d_y.data_ptr()
    assert L.qpsk_agc_process_dev(agc._h, x0, y0, 3, 2 * n, 2 * n, None) == N.ERR_ARG            # odd count
    assert L.qpsk_agc_process_dev(agc._h, x0, y0, 2 * n, 2 * n + 1, 2 * n, None) == N.ERR_ARG    # odd stride
    assert L.qpsk_agc_process_dev(agc._h, x0, y0, 2 * n, 2 * n - 2, 2 * n, None) == N.ERR_ARG    # rows overlap
    assert L.qpsk_agc_process_dev(agc._h, x0, y0, 2 * n, 2 * n, 2 * n - 2, None) == N.ERR_CAPACITY
    assert L.qpsk_agc_process_dev(agc._h, x0 + 4, y0, 2 * n, 2 * n, 2 * n, None) == N.ERR_ARG    # 4-byte aligned
    assert L.qpsk_agc_process_dev(agc._h, x0, None, 2 * n, 2 * n, 2 * n, None) == N.ERR_NULL
    assert L.qpsk_agc_process_dev(agc._h, x0, y0, -2, 2 * n, 2 * n, None) == N.ERR_RANGE
    assert L.qpsk_agc_process_dev(None, x0, y0, 2 * n, 2 * n, 2 * n, None) == N.ERR_NULL
    assert L.qpsk_agc_process_dev(agc._h, None, None, 0, 0, 0, None) == N.OK                     # empty call
    g = np.zeros(C, np.float32)
    assert L.qpsk_agc_gain(agc._h, g.ctypes.data_as(N.f32p), C - 1) == N.ERR_CAPACITY
    assert np.all(agc.gain == np.float32(65536.0))                                                 # before any sample
    agc.process_dev(x0, y0, 2 * n, stream=0)
    torch.cuda.synchronize()
    got = d_y[: C * 2 * n].cpu().numpy().view(np.complex64).reshape(C, n)
    assert np.array_equal(_bits(got), _bits(want))
    d_g = torch.zeros(C, dtype=torch.float32, device="cuda")
    agc.gain_dev(d_g.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(_bits(d_g.cpu().numpy()), _bits(agc.gain))


def test_power_of_two_levels_give_identical_bits(gpu):
    rng = np.random.default_rng(11)
    C, n = 16, 6000
    mag = 10.0 ** rng.uniform(-1, 1, (C, n))
    x = (mag * np.exp(2j * np.pi * rng.uniform(0, 1, (C, n)))).astype(np.complex64)
    for W in (1, 31, 64, 1000):
        want = gpu.Agc(W, 1.0, 1e6, C).process(x)
        assert np.array_equal(_bits(want), _bits(AgcBatch(W, 1.0, 1e6, C).process(x)))
        for k in range(-10, 7):
            xs = (x * np.float32(2.0 ** k)).astype(np.complex64)
            assert np.array_equal(_bits(gpu.Agc(W, 1.0, 1e6, C).process(xs)), _bits(want)), (W, k)


# ---- demodulator stage ---------------------------------------------------------------------------------------------
def _scene_batch(orc, C, n_total, seed=5):
    """C rows cycling over the six DDC-scene carriers (CPU bank), row r at level 2^(r mod 11 - 7), each with a residual
    offset of 0.001 cycles per sample, zero-padded to n_total samples."""
    from ddc_oracle import DdcPoly
    h = scene_taps()
    wide, pays = ddc_scene(orc, h, SCENE_D, SCENE_FREQS, seed=seed)
    y = DdcPoly(h, SCENE_FREQS, SCENE_D).process(wide)
    rot = np.exp(2j * np.pi * 0.001 * np.arange(y.shape[1]))
    rows = np.zeros((C, n_total), np.complex64)
    for r in range(C):
        rows[r, : y.shape[1]] = (y[r % len(pays)] * rot * 2.0 ** (r % 11 - 7)).astype(np.complex64)
    return rows, [pays[r % len(pays)] for r in range(C)]


# W = 4096 with the FLL: the first 4200-sample call runs the time-chunk pipeline and the AGC's discard takes its first five
# chunks whole and part of the sixth
@pytest.mark.parametrize("use_fll,W", [(False, 64), (True, 64), (True, 4096)], ids=["False", "True", "True-W4096"])
def test_demod_stage_matches_oracle(gpu, orc, use_fll, W):
    C = 256
    if W == 64:
        rows, pays = _scene_batch(orc, C, 4200)       # 4200 samples: with the FLL on, the time-chunk pipeline runs
        cuts = [0, 30, 1500, 4200]                    # the first call is shorter than the AGC's discard
    else:
        rows, pays = _scene_batch(orc, C, 3 * 4200)
        cuts = [0, 4200, 8400, 12600]
    dem = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, use_fll=use_fll, channels=C)
    dem.set_agc(W, 1.0, 65536.0)
    ref = AgcDemod(orc, SCENE_FS, SCENE_RS, 0.35, 10, channels=C, tsc=TSC, use_fll=use_fll)
    ref.set_agc(W, 1.0, 65536.0)
    for a, b in zip(cuts[:-1], cuts[1:]):
        part = np.ascontiguousarray(rows[:, a:b]).view(np.float32)
        assert dem.DeModulate(part) == ref.DeModulate(part), (a, b)
    # host rows, cf32 and CS16, through the same calls: the payloads of the oracle on the values the device widens to
    scale = float(np.float32(np.abs(rows.view(np.float32)).max() / 30000.0))
    x16 = np.clip(np.round(rows.view(np.float32) / scale), -32768, 32767).astype(np.int16)
    xf = (x16.astype(np.float32) * np.float32(scale)).astype(np.float32)
    d32, d16 = (gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, use_fll=use_fll, channels=C) for _ in range(2))
    ref = AgcDemod(orc, SCENE_FS, SCENE_RS, 0.35, 10, channels=C, tsc=TSC, use_fll=use_fll)
    for d in (d32, d16, ref):
        d.set_agc(W, 1.0, 65536.0)
    for a, b in zip(cuts[:-1], cuts[1:]):
        want = ref.DeModulateBytes(np.ascontiguousarray(xf[:, 2 * a: 2 * b]), b"START", b"END")
        assert d32.DeModulateBytes(np.ascontiguousarray(xf[:, 2 * a: 2 * b]), b"START", b"END") == want, (a, b)
        assert d16.DeModulateBytesCs16(np.ascontiguousarray(x16[:, 2 * a: 2 * b]), scale, b"START", b"END") == want, (a, b)
    # the frames decode at every level
    if W == 64:
        dem2 = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, use_fll=use_fll, channels=C)
        dem2.set_agc(W, 1.0, 65536.0)
        got = dem2.DeModulateBytes(np.ascontiguousarray(rows).view(np.float32), b"START", b"END")
        assert got == pays


# The profiler runs in a child process: once a torch.profiler session has been opened in the pytest process, the profiled
# tests of other files that run later in the same process recorded no kernels at all.
_PROFILE_CHILD = """
import sys
sys.path[:0] = {paths!r}
import numpy as np
import qpsk_modulator_demodulator_b200 as Q
from symsync_dispatch import launched_kernels
Q.set_device({device})
x = np.random.default_rng(1).standard_normal((256, 6000)).astype(np.float32)
d = Q.QPSKDeModulator(4000, 1000, 0.35, 10, tsc={tsc!r}, use_fll={use_fll}, channels=256)
d.set_agc(64)
d.DeModulate(np.ascontiguousarray(x[:, :400]))      # past the AGC's discard
_, names = launched_kernels(lambda: d.DeModulate(x))
print("KERNELS", repr(sorted(set(names))))
"""


@pytest.mark.parametrize("use_fll", [False, True])
def test_profiler_shows_the_fused_symbol_stage_with_the_stage_on(gpu, use_fll):
    """256 channels of 3000 samples (with the FLL: the time-chunk pipeline): the AGC and the fused symbol-stage kernel
    both run."""
    import ast
    import os
    import subprocess
    import sys
    here = os.path.dirname(os.path.abspath(__file__))
    code = _PROFILE_CHILD.format(paths=[os.path.dirname(here), here], device=int(os.environ.get("LOCAL_RANK", "0")),
                                 tsc=TSC, use_fll=use_fll)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("KERNELS ")][-1]
    names = ast.literal_eval(line[len("KERNELS "):])
    assert any("agc_block_kernel" in k for k in names), names
    assert symsync_variants(names), names


def test_demod_stage_off_is_the_plain_chain_and_set_resets_only_the_stage(gpu, orc):
    C = 33
    rows, _ = _scene_batch(orc, C, 3000)
    x = np.ascontiguousarray(rows).view(np.float32)
    plain = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, channels=C).DeModulate(x)
    dem = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, channels=C)
    dem.set_agc(16)
    dem.set_agc(0)
    assert dem.DeModulate(x) == plain
    from qpsk_modulator_demodulator_b200 import _native as N
    with pytest.raises(N.QpskCudaError):
        dem.set_agc(5000)
    with pytest.raises(N.ArgumentOutOfRangeException):
        dem.set_agc(16, 0.0)
    # a fresh stage mid-stream: the rest of the stream goes through a new AGC, the loops keep their state
    half = 1400
    a = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, channels=C)
    b = AgcDemod(orc, SCENE_FS, SCENE_RS, 0.35, 10, channels=C)
    x1, x2 = np.ascontiguousarray(rows[:, :half]).view(np.float32), np.ascontiguousarray(rows[:, half:]).view(np.float32)
    a.set_agc(8)
    b.set_agc(8)
    assert a.DeModulate(x1) == b.DeModulate(x1)
    a.set_agc(32, 2.0, 100.0)
    b.set_agc(32, 2.0, 100.0)
    assert a.DeModulate(x2) == b.DeModulate(x2)


def test_ddc_rows_feed_the_demodulator_with_the_stage_on_one_stream(gpu, orc):
    import torch
    h = scene_taps()
    K = len(SCENE_FREQS)
    wide, pays = ddc_scene(orc, h, SCENE_D, SCENE_FREQS, seed=9)
    wide = wide * 2.0 ** -6                                          # every carrier 36 dB down
    bank = gpu.DdcBank(h, SCENE_FREQS, SCENE_D)
    dem = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, channels=K)
    dem.set_agc(32)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        d_x = torch.from_numpy(wide.astype(np.complex64).view(np.float32).copy()).cuda()
        n_out = wide.size // SCENE_D
        stride = 2 * n_out + 64
        d_y = torch.zeros((K, stride), dtype=torch.float32, device="cuda")
        cap = 256
        d_pay = torch.zeros((K, cap), dtype=torch.uint8, device="cuda")
        d_n = torch.zeros(K, dtype=torch.int64, device="cuda")
        nf = bank.process_dev(d_x.data_ptr(), d_x.numel(), d_y.data_ptr(), stride, ts.cuda_stream)
        assert nf == 2 * n_out
        dem.demod_bytes_dev(d_y.data_ptr(), nf, stride, b"START", b"END", d_pay.data_ptr(), cap, d_n.data_ptr(), ts.cuda_stream)
        ts.synchronize()
        pay, nb = d_pay.cpu().numpy(), d_n.cpu().numpy()
    for k in range(K):
        assert pay[k, : nb[k]].tobytes() == pays[k], k
