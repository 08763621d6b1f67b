"""GPU: the digital down-converter bank (csrc/ddc.cu) against the fp64 rotated-tap restatement (tests/ddc_oracle.py)
within 1e-5 max|y| over both kernel shapes; bit-identical outputs for any chunking, for the host and device entry points
and after reset(); untouched guard bands; argument checks; agreement with the PFB channelizer on a full grid and with the
full bank on a subset; 64-bit counters and output indices; and an off-grid QPSK scene demodulated straight from the
bank's output rows."""
import ctypes as C

import numpy as np
import pytest

from ddc_oracle import (SCENE_D, SCENE_FREQS, SCENE_FS, SCENE_RS, TSC, DdcPoly, ddc_scene, phase_angle, phase_word,
                        scene_taps)

pytestmark = pytest.mark.gpu

SMALL_K = 8                      # csrc/ddc.cu kDdcSmallK: K <= 8 runs the 4-channel x 1024-output shape
TILE = {True: 1024, False: 128}  # outputs per CTA of the two shapes


def _cx64(rng, n):
    return (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)


def _freqs(rng, K):
    return list(rng.uniform(-0.5, 0.5, K))


def _check(got, want):
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.abs(got.astype(np.complex128) - want).max() <= 1e-5 * np.abs(want).max()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# K = 1, odd K, both sides of the shape switch, K not a multiple of either channel block, K = 2048; D = 1, odd D and powers
# of two up to 1024; N < D, N not a multiple of D, N = 4096
@pytest.mark.parametrize("K,D,N", [(1, 1, 1), (1, 2, 4096), (3, 3, 10), (5, 5, 2), (8, 7, 100), (9, 16, 128), (33, 1, 33),
                                   (33, 64, 300), (17, 256, 4096), (2048, 4, 64), (4, 1024, 4096), (40, 1024, 100),
                                   (7, 512, 37), (64, 8, 4096), (100, 32, 31)])
def test_matches_rotated_tap_oracle(gpu, K, D, N):
    rng = np.random.default_rng(K * 100000 + D * 100 + N)
    h = (rng.standard_normal(N) / np.sqrt(N)).astype(np.float32)
    freqs = _freqs(rng, K)
    n_out = 2 * TILE[K <= SMALL_K] + 37 if K < 1000 else 300      # more than two tiles, ragged end
    x = _cx64(rng, n_out * D + D // 2 + 1)
    got = gpu.DdcBank(h, freqs, D).process(x)
    _check(got, DdcPoly(h, freqs, D).process(x))


@pytest.mark.parametrize("K,D,N", [(3, 16, 100), (40, 7, 64), (5, 1024, 300), (33, 1, 9)])
def test_any_chunking_host_and_device_paths_and_reset_are_bit_identical(gpu, K, D, N):
    import torch
    rng = np.random.default_rng(7 + K + D)
    h = rng.standard_normal(N)
    freqs = _freqs(rng, K)
    x = _cx64(rng, 300 * D + 5)
    one = gpu.DdcBank(h, freqs, D)
    ref = one.process(x)
    _check(ref, DdcPoly(h.astype(np.float32), freqs, D).process(x))
    one.reset()
    assert np.array_equal(_bits(one.process(x)), _bits(ref))
    # random chunks: odd sizes, sizes below D, empty calls
    ch = gpu.DdcBank(h, freqs, D)
    cuts, a = [], 0
    while a < x.size:
        c = int(rng.choice([0, 1, 3, max(D - 1, 0), D + 1, 2 * D + 7, int(rng.integers(0, 40 * D))]))
        cuts.append(min(c, x.size - a))
        a += cuts[-1]
    starts = np.cumsum([0] + cuts[:-1])
    got = np.concatenate([ch.process(x[b:b + c]) for b, c in zip(starts, cuts)], axis=1)
    assert np.array_equal(_bits(got), _bits(ref))
    # device path, the same chunks at odd sample offsets into one buffer, all on one user stream
    dv = gpu.DdcBank(h, freqs, D)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        d_x = torch.from_numpy(x.view(np.float32).copy()).cuda()
        stride = 2 * (x.size // D + 4)
        d_y = torch.full((K, stride), 7.0, dtype=torch.float32, device="cuda")
        col = 0
        for b, c in zip(starts, cuts):
            col += dv.process_dev(d_x.data_ptr() + 8 * int(b), 2 * c, d_y.data_ptr() + 4 * col, stride, ts.cuda_stream)
        ts.synchronize()                                        # reset waits for the handle's own stream only
        dv.reset()
        d_y2 = torch.full((K, stride), 7.0, dtype=torch.float32, device="cuda")
        nf = dv.process_dev(d_x.data_ptr(), 2 * x.size, d_y2.data_ptr(), stride, ts.cuda_stream)
        ts.synchronize()
        y, y2 = d_y.cpu().numpy(), d_y2.cpu().numpy()
    assert col == nf == 2 * ref.shape[1]
    assert np.array_equal(_bits(np.ascontiguousarray(y[:, :col]).view(np.complex64)), _bits(ref))
    assert np.array_equal(_bits(np.ascontiguousarray(y2[:, :nf]).view(np.complex64)), _bits(ref))
    assert np.all(y[:, col:] == 7.0)


@pytest.mark.parametrize("K", [5, 50])
def test_guard_bands_and_row_padding_untouched_and_repeatable(gpu, K):
    import torch
    D, N = 16, 128
    rng = np.random.default_rng(11 + K)
    h = scene_taps(D, 8)
    freqs = _freqs(rng, K)
    x = _cx64(rng, 3000 * D + 17)
    n_out = x.size // D
    stride = 2 * n_out + 6
    guard = 4096
    ts = torch.cuda.Stream()
    outs = []
    for _ in range(2):
        with torch.cuda.stream(ts):
            d_x = torch.from_numpy(x.view(np.float32).copy()).cuda()
            buf = torch.full((guard + K * stride + guard,), -3.5, dtype=torch.float32, device="cuda")
            p = gpu.DdcBank(h, freqs, D)
            nf = p.process_dev(d_x.data_ptr(), 2 * x.size, buf.data_ptr() + 4 * guard, stride, ts.cuda_stream)
            ts.synchronize()
            b = buf.cpu().numpy()
        assert nf == 2 * n_out
        assert np.all(b[:guard] == -3.5) and np.all(b[guard + K * stride:] == -3.5)
        rows = b[guard:guard + K * stride].reshape(K, stride)
        assert np.all(rows[:, nf:] == -3.5)
        outs.append(rows[:, :nf].copy())
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32))
    _check(np.ascontiguousarray(outs[0]).view(np.complex64), DdcPoly(h.astype(np.float32), freqs, D).process(x))


def test_argument_checks(gpu):
    L = gpu._native.lib()
    N = gpu._native
    h = np.ones(64, np.float32) / 64
    hp = h.ctypes.data_as(N.f32p)
    f = np.zeros(2049, np.float64)
    fp = f.ctypes.data_as(N.f64p)
    out = C.c_void_p()

    def create(taps=hp, n=64, freqs=fp, K=4, D=8):
        return L.qpsk_ddc_create(taps, n, freqs, K, D, C.byref(out))

    assert create(K=0) == N.ERR_UNSUPPORTED and create(K=2049) == N.ERR_UNSUPPORTED
    assert create(D=0) == N.ERR_UNSUPPORTED and create(D=1025) == N.ERR_UNSUPPORTED
    big = np.ones(4097, np.float32)
    assert create(taps=big.ctypes.data_as(N.f32p), n=4097) == N.ERR_UNSUPPORTED
    assert create(n=0) == N.ERR_ARG and create(n=-3) == N.ERR_ARG
    assert create(taps=None) == N.ERR_NULL and create(freqs=None) == N.ERR_NULL
    assert L.qpsk_ddc_create(hp, 64, fp, 4, 8, None) == N.ERR_NULL
    for v in (np.inf, -np.inf, np.nan):
        bad = h.copy()
        bad[5] = v
        assert create(taps=bad.ctypes.data_as(N.f32p)) == N.ERR_RANGE
    for v in (0.5, 0.75, -0.5000001, np.inf, np.nan):
        bf = np.zeros(4)
        bf[2] = v
        assert create(freqs=bf.ctypes.data_as(N.f64p)) == N.ERR_RANGE, v
    for good in (dict(K=1, D=1, n=1), dict(K=2048, D=1024, n=64)):
        st = create(**good)
        assert st == N.OK, good
        L.qpsk_ddc_destroy(out)
    bf = np.array([-0.5, 0.0, 0.5 - 2 ** -53, 0.25])
    assert create(freqs=bf.ctypes.data_as(N.f64p)) == N.OK
    L.qpsk_ddc_destroy(out)
    with pytest.raises(gpu.ArgumentNullException):
        gpu.DdcBank(None, [0.1], 4)
    with pytest.raises(gpu.ArgumentNullException):
        gpu.DdcBank(h, None, 4)
    # odd n_floats -> ARG; a too-small stride -> CAPACITY with the needed size, and nothing consumed
    D = 16
    rng = np.random.default_rng(3)
    hh = rng.standard_normal(5 * D + 3)
    freqs = [0.01, -0.2, 0.33]
    x = _cx64(rng, 40 * D + 3)
    xf = x.view(np.float32)
    p = gpu.DdcBank(hh, freqs, D)
    want = gpu.DdcBank(hh, freqs, D).process(x)
    n = C.c_int64(0)
    y = np.zeros((3, 200), np.float32)
    assert L.qpsk_ddc_process(p._h, xf.ctypes.data, 7, y.ctypes.data, 200, C.byref(n)) == N.ERR_ARG
    a = 11 * D + 5                                              # first call leaves 5 samples pending
    first = p.process(x[:a])
    assert L.qpsk_ddc_process(p._h, xf[2 * a:].ctypes.data, 2 * (x.size - a), y.ctypes.data, 2, C.byref(n)) == N.ERR_CAPACITY
    assert n.value == 2 * ((x.size - a + 5) // D)
    assert L.qpsk_ddc_process_dev(p._h, 0, 2 * (x.size - a), 0, 2, C.byref(n), None) == N.ERR_CAPACITY
    rest = p.process(x[a:])
    assert np.array_equal(_bits(np.concatenate([first, rest], axis=1)), _bits(want))
    assert L.qpsk_ddc_process_dev(p._h, 0, 3, 0, 64, C.byref(n), None) == N.ERR_ARG
    assert L.qpsk_ddc_process_dev(p._h, 0, 4, 0, 63, C.byref(n), None) == N.ERR_ARG


@pytest.mark.parametrize("M", [16, 64])
def test_full_grid_matches_the_pfb_channelizer_and_a_subset_gives_its_rows(gpu, M):
    rng = np.random.default_rng(M)
    h = gpu.pfb_taps(M, 8, 0.5 / M, 60.0)
    x = _cx64(rng, 700 * M + 9)
    freqs = [(k if k < M // 2 else k - M) / M for k in range(M)]
    full = gpu.DdcBank(h, freqs, M).process(x)
    pfb = gpu.PfbChannelizer(h, M).process(x).astype(np.complex128) * np.exp(2j * np.pi * np.arange(M) / M)[:, None]
    assert full.shape == pfb.shape
    assert np.abs(full - pfb).max() <= 1e-5 * np.abs(pfb).max()
    pick = [3, M // 2, 1, M - 1, 7]
    sub = gpu.DdcBank(h, [freqs[k] for k in pick], M).process(x)
    assert np.array_equal(_bits(sub), _bits(full[pick]))


def test_counter_past_2_pow_32_samples(gpu):
    import torch
    K, D, N = 3, 1024, 64
    rng = np.random.default_rng(21)
    h = rng.standard_normal(N).astype(np.float32)
    freqs = [0.1234567, -0.4999, 2.0 ** -40]
    bank = gpu.DdcBank(h, freqs, D)
    ts = torch.cuda.Stream()
    chunk = 1 << 28
    with torch.cuda.stream(ts):
        zeros = torch.zeros(2 * chunk, dtype=torch.float32, device="cuda")
        stride = 2 * (chunk // D)
        d_y = torch.empty((K, stride), dtype=torch.float32, device="cuda")
        for _ in range(16):
            assert bank.process_dev(zeros.data_ptr(), 2 * chunk, d_y.data_ptr(), stride, ts.cuda_stream) == stride
        x = _cx64(rng, 300 * D + 77)
        d_x = torch.from_numpy(x.view(np.float32).copy()).cuda()
        nf = bank.process_dev(d_x.data_ptr() + 8, 2 * (x.size - 1), d_y.data_ptr(), stride, ts.cuda_stream)
        ts.synchronize()
        y = np.ascontiguousarray(d_y.cpu().numpy()[:, :nf]).view(np.complex64)
    want = DdcPoly(h, freqs, D, start=16 * chunk).process(x[1:])
    _check(y, want)


def test_one_call_whose_output_spans_more_than_2_pow_31_floats(gpu):
    import torch
    K, D, N = 2048, 1024, 64
    n = 1 << 30
    n_out = n // D
    assert K * 2 * n_out > 2 ** 31
    rng = np.random.default_rng(5)
    h = rng.standard_normal(N).astype(np.float32)
    freqs = _freqs(rng, K)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        g = torch.Generator(device="cuda").manual_seed(17)
        d_x = torch.randn(2 * n, dtype=torch.float32, device="cuda", generator=g)
        d_y = torch.empty((K, 2 * n_out), dtype=torch.float32, device="cuda")
        nf = gpu.DdcBank(h, freqs, D).process_dev(d_x.data_ptr(), 2 * n, d_y.data_ptr(), 2 * n_out, ts.cuda_stream)
        ts.synchronize()
        assert nf == 2 * n_out
        pts = [(K - 1, n_out - 1), (0, 0), (K - 1, 0), (0, n_out - 1), (1234, n_out // 2)]
        pts += [(int(rng.integers(0, K)), int(rng.integers(0, n_out))) for _ in range(59)]
        got, want = [], []
        for k, m in pts:
            nm = m * D + D - 1
            lo = max(0, nm - (N - 1))
            win = d_x[2 * lo: 2 * (nm + 1)].cpu().numpy().view(np.complex64).astype(np.complex128)
            idx = np.arange(lo, nm + 1)
            i = nm - idx
            with np.errstate(over="ignore"):
                rot = np.exp(-1j * phase_angle(phase_word(freqs[k]), idx))
            want.append(np.sum(h[i].astype(np.float64) * win * rot))
            got.append(complex(*d_y[k, 2 * m: 2 * m + 2].cpu().numpy()))
    got, want = np.array(got), np.array(want)
    assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()


def test_off_grid_scene_feeds_the_batch_demodulator(gpu, orc):
    import torch
    h = scene_taps()
    K = len(SCENE_FREQS)
    wide, pays = ddc_scene(orc, h, SCENE_D, SCENE_FREQS, seed=9)
    bank = gpu.DdcBank(h, SCENE_FREQS, SCENE_D)
    dem = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, channels=K)
    # one user stream orders the buffer fills, the bank and the demodulator
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
        pay, nb, rows = d_pay.cpu().numpy(), d_n.cpu().numpy(), d_y.cpu().numpy()[:, :nf]
    for k in range(K):
        assert pay[k, : nb[k]].tobytes() == pays[k], k
    _check(np.ascontiguousarray(rows).view(np.complex64), DdcPoly(h.astype(np.float32), SCENE_FREQS, SCENE_D).process(wide.astype(np.complex64)))
