"""GPU: the rational resampler (csrc/resamp.cu) against the fp64 polyphase restatement (tests/resamp_oracle.py) within
1e-5 max|y| over both kernel shapes, every ratio of the CPU tests and P = 1, 2, 63, 64; every compiled resamp_kernel
instantiation listed from the library and seen running in the profiler; bit-identical outputs for any chunking, for the
host and device entry points, strided and offset rows, after reset(), on repeat runs and for a subset of channels against
the full batch; untouched guard bands; argument checks; 64-bit counters and output indices; a transmit round trip through
5/8 and 8/5; and a receive chain DdcBank -> Resampler -> QPSKDeModulator on one stream at 4.096 samples per symbol."""
import ctypes as C
import os

import numpy as np
import pytest

import kernel_variants as kv
from ddc_oracle import TSC, scene_taps
from resamp_oracle import (SCENE_D, SCENE_FREQS, SCENE_FS, SCENE_L, SCENE_M, SCENE_RS, ResampPoly, resamp_count,
                           resamp_scene, resamp_taps)

pytestmark = pytest.mark.gpu

SMALL_K = 8                      # csrc/resamp.cu kResampSmallK: K <= 8 runs the one-channel x 256-output shape
TILE = {True: 256, False: 32}    # outputs per CTA of the two shapes
SHAPES = {True: "resamp_kernel<1, 1, 1, 2048>", False: "resamp_kernel<32, 2, 4, 64>"}


def _cx64(rng, *shape):
    return (rng.standard_normal(shape) + 1j * rng.standard_normal(shape)).astype(np.complex64)


def _check(got, want):
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.abs(got.astype(np.complex128) - want).max() <= 1e-5 * np.abs(want).max()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _n_in_for(L, M, n_out):
    """Inputs that complete at least n_out outputs."""
    return -(-n_out * M // L) + 1


# (K, L, M, N): every ratio; K = 1, 8 | 9 (both sides of the shape switch), odd K, K not a multiple of the 64-channel
# block, K = 16384; P = 1, 2, 63, 64; N < L and N not a multiple of L
CASES = [(1, 1, 1, 1), (1, 5, 8, 120), (8, 8, 5, 63 * 8), (9, 8, 5, 64 * 8), (3, 1, 4, 63), (65, 4, 1, 2 * 4),
         (33, 125, 128, 3000), (1, 1024, 1023, 16 * 1024 - 5), (7, 3, 1024, 190), (100, 1024, 1023, 700), (2, 64, 3, 1),
         (64, 5, 8, 64 * 5), (130, 1, 1, 64), (16384, 5, 8, 40), (5, 1, 1024, 64), (200, 2, 1, 3)]


@pytest.mark.parametrize("K,L,M,N", CASES)
def test_matches_polyphase_oracle(gpu, K, L, M, N):
    rng = np.random.default_rng(K * 100003 + L * 1009 + M * 17 + N)
    h = (rng.standard_normal(N) / np.sqrt(max(1, N // L))).astype(np.float32)
    n_out = 2 * TILE[K <= SMALL_K] + 37 if K < 1000 else 70       # more than two tiles, ragged end
    x = _cx64(rng, K, _n_in_for(L, M, n_out))
    got = gpu.Resampler(h, L, M, K).process(x)
    want = ResampPoly(h, L, M, K).process(x)
    assert got.shape[1] == resamp_count(x.shape[1], L, M)
    _check(got, want)


def test_every_instantiation_is_compiled_tested_and_runs(gpu):
    """The instantiations in the library are exactly the two shapes the parity cases reach, and the profiler (in a child
    process) sees the predicted one run for every call of the resampler rows in tests/kernel_variants.py."""
    got = kv.compiled(gpu._native.LIB_PATH)["resamp"]
    assert got == set(SHAPES.values()), got
    assert {SHAPES[K <= SMALL_K] for K, _, _, _ in CASES} == got
    ran = kv.launched_in_child("resamp", int(os.environ.get("LOCAL_RANK", "0")))
    assert ran == kv.predicted_launches("resamp") and set(ran) == got, ran


@pytest.mark.parametrize("K,L,M,N", [(3, 5, 8, 100), (40, 8, 5, 300), (5, 1, 1024, 64), (70, 125, 128, 1000),
                                     (2, 1024, 1023, 3000)])
def test_chunking_offsets_strides_reset_repeat_and_subset_are_bit_identical(gpu, K, L, M, N):
    import torch
    rng = np.random.default_rng(K + L + M + N)
    h = rng.standard_normal(N).astype(np.float32)
    n = _n_in_for(L, M, 700)
    x = _cx64(rng, K, n)
    one = gpu.Resampler(h, L, M, K)
    ref = one.process(x)
    _check(ref, ResampPoly(h, L, M, K).process(x))
    one.reset()
    assert np.array_equal(_bits(one.process(x)), _bits(ref))
    # host path, random chunks: empty calls, one-sample calls, calls shorter than M / L
    cuts, a = [], 0
    while a < n:
        c = int(rng.choice([0, 1, 1, max(M // L - 1, 0), M // L + 1, int(rng.integers(0, 40 * max(1, M // L)))]))
        cuts.append(min(c, n - a))
        a += cuts[-1]
    starts = np.cumsum([0] + cuts[:-1])
    ch = gpu.Resampler(h, L, M, K)
    got = np.concatenate([ch.process(np.ascontiguousarray(x[:, b:b + c])).reshape(K, -1) for b, c in zip(starts, cuts)],
                         axis=1)
    assert np.array_equal(_bits(got), _bits(ref))
    # device path: the same chunks read at odd sample offsets of rows with a stride past the row, into strided rows
    ldx = 2 * n + 6
    xin = np.zeros((K, ldx + 2), np.float32)
    xin[:, 2:2 + 2 * n] = x.view(np.float32)
    ldy = 2 * ref.shape[1] + 10
    dv = gpu.Resampler(h, L, M, K)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        d_x = torch.from_numpy(xin.copy()).cuda()
        for rep in range(2):
            d_y = torch.full((K, ldy), 7.0, dtype=torch.float32, device="cuda")
            col = 0
            for b, c in zip(starts, cuts):
                col += dv.process_dev(d_x.data_ptr() + 4 * (2 + 2 * int(b)), 2 * c, d_y.data_ptr() + 4 * col, ldy,
                                      in_stride=ldx + 2, stream=ts.cuda_stream)
            ts.synchronize()
            y = d_y.cpu().numpy()
            assert col == 2 * ref.shape[1]
            assert np.array_equal(_bits(np.ascontiguousarray(y[:, :col]).view(np.complex64)), _bits(ref)), rep
            assert np.all(y[:, col:] == 7.0)
            dv.reset()
    # a subset of the rows, and each row on its own handle, give the rows of the full batch
    pick = [K - 1, 0] + ([K // 2] if K > 2 else [])
    sub = gpu.Resampler(h, L, M, len(pick)).process(np.ascontiguousarray(x[pick]))
    assert np.array_equal(_bits(sub), _bits(ref[pick]))
    row = gpu.Resampler(h, L, M, 1).process(np.ascontiguousarray(x[K - 1]))
    assert np.array_equal(_bits(row), _bits(ref[K - 1]))


@pytest.mark.parametrize("K", [5, 50])
def test_guard_bands_untouched(gpu, K):
    import torch
    L, M, N = 5, 8, 200
    rng = np.random.default_rng(11 + K)
    h = resamp_taps(L, M, 40).astype(np.float32)
    x = _cx64(rng, K, 3000)
    n_out = resamp_count(x.shape[1], L, M)
    stride, guard = 2 * n_out + 6, 4096
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        d_x = torch.from_numpy(x.view(np.float32).copy()).cuda()
        buf = torch.full((guard + K * stride + guard,), -3.5, dtype=torch.float32, device="cuda")
        nf = gpu.Resampler(h, L, M, K).process_dev(d_x.data_ptr(), 2 * x.shape[1], buf.data_ptr() + 4 * guard, stride,
                                                   stream=ts.cuda_stream)
        ts.synchronize()
        b = buf.cpu().numpy()
    assert nf == 2 * n_out
    assert np.all(b[:guard] == -3.5) and np.all(b[guard + K * stride:] == -3.5)
    rows = b[guard:guard + K * stride].reshape(K, stride)
    assert np.all(rows[:, nf:] == -3.5)
    _check(np.ascontiguousarray(rows[:, :nf]).view(np.complex64), ResampPoly(h, L, M, K).process(x))


def test_argument_checks_and_refused_calls_consume_nothing(gpu):
    import torch
    N = gpu._native
    L_ = N.lib()
    h = np.ones(64, np.float32) / 64
    hp = h.ctypes.data_as(N.f32p)
    out = C.c_void_p()

    def create(taps=hp, n=64, L=4, M=8, K=4):
        return L_.qpsk_resamp_create(taps, n, L, M, K, C.byref(out))

    for bad in (dict(K=0), dict(K=16385), dict(L=0), dict(L=1025), dict(M=0), dict(M=1025), dict(n=65, L=1)):
        assert create(**bad) == N.ERR_UNSUPPORTED, bad
    big = np.ones(16385, np.float32)
    assert create(taps=big.ctypes.data_as(N.f32p), n=16385, L=1024) == N.ERR_UNSUPPORTED
    assert create(n=0) == N.ERR_ARG and create(n=-3) == N.ERR_ARG
    assert create(taps=None) == N.ERR_NULL
    assert L_.qpsk_resamp_create(hp, 64, 4, 8, 4, None) == N.ERR_NULL
    for v in (np.inf, -np.inf, np.nan):
        bad = h.copy()
        bad[5] = v
        assert create(taps=bad.ctypes.data_as(N.f32p)) == N.ERR_RANGE
    full = np.ones(16384, np.float32)
    for good in (dict(K=1, L=1, M=1, n=1), dict(K=16384, L=1024, M=1024, n=64), dict(L=256, n=16384, taps=full.ctypes.data_as(N.f32p))):
        assert create(**good) == N.OK, good
        L_.qpsk_resamp_destroy(out)
    with pytest.raises(gpu.ArgumentNullException):
        gpu.Resampler(None, 1, 1)
    # CAPACITY with the needed count, nothing consumed; odd counts and strides, overlap, alignment -> ARG
    K, L, M = 3, 5, 8
    rng = np.random.default_rng(3)
    hh = rng.standard_normal(37).astype(np.float32)
    x = _cx64(rng, K, 777)
    want = gpu.Resampler(hh, L, M, K).process(x)
    p = gpu.Resampler(hh, L, M, K)
    first = p.process(np.ascontiguousarray(x[:, :101]))
    rest = np.ascontiguousarray(x[:, 101:])
    n = C.c_int64(0)
    y = np.zeros((K, 4), np.float32)
    assert L_.qpsk_resamp_process(p._h, rest.ctypes.data, 2 * rest.shape[1], y.ctypes.data, 4, C.byref(n)) == N.ERR_CAPACITY
    assert n.value == 2 * (resamp_count(777, L, M) - resamp_count(101, L, M))
    assert L_.qpsk_resamp_process(p._h, rest.ctypes.data, 7, y.ctypes.data, 400, C.byref(n)) == N.ERR_ARG
    assert L_.qpsk_resamp_process(p._h, rest.ctypes.data, -2, y.ctypes.data, 400, C.byref(n)) == N.ERR_RANGE
    d_x = torch.from_numpy(rest.view(np.float32).copy()).cuda()
    nf = 2 * rest.shape[1]
    d_y = torch.zeros(K * 2000 + 2, dtype=torch.float32, device="cuda")
    x0, y0 = d_x.data_ptr(), d_y.data_ptr()
    assert L_.qpsk_resamp_process_dev(p._h, x0, nf, nf, y0, 4, C.byref(n), None) == N.ERR_CAPACITY
    assert L_.qpsk_resamp_process_dev(p._h, x0, 3, 4, y0, 2000, C.byref(n), None) == N.ERR_ARG          # odd count
    assert L_.qpsk_resamp_process_dev(p._h, x0, nf, nf + 1, y0, 2000, C.byref(n), None) == N.ERR_ARG    # odd stride
    assert L_.qpsk_resamp_process_dev(p._h, x0, nf, nf, y0, 2001, C.byref(n), None) == N.ERR_ARG
    assert L_.qpsk_resamp_process_dev(p._h, x0, nf, nf - 2, y0, 2000, C.byref(n), None) == N.ERR_ARG    # rows overlap
    assert L_.qpsk_resamp_process_dev(p._h, x0 + 4, nf, nf, y0, 2000, C.byref(n), None) == N.ERR_ARG    # 4-byte aligned
    assert L_.qpsk_resamp_process_dev(p._h, x0, nf, nf, x0 + 8 * nf, 2000, C.byref(n), None) == N.ERR_ARG  # out over in
    assert L_.qpsk_resamp_process_dev(p._h, x0, nf, nf, None, 2000, C.byref(n), None) == N.ERR_NULL
    assert L_.qpsk_resamp_process_dev(p._h, x0, -2, nf, y0, 2000, C.byref(n), None) == N.ERR_RANGE
    assert L_.qpsk_resamp_process_dev(None, x0, nf, nf, y0, 2000, C.byref(n), None) == N.ERR_NULL
    assert L_.qpsk_resamp_process_dev(p._h, x0, nf, nf, y0, 2000, None, None) == N.ERR_NULL
    assert L_.qpsk_resamp_process_dev(p._h, None, 0, 0, None, 0, C.byref(n), None) == N.OK and n.value == 0
    got = p.process(rest)
    assert np.array_equal(_bits(np.concatenate([first, got], axis=1)), _bits(want))


def test_counter_past_2_pow_32_samples(gpu):
    import torch
    K, L, M, N = 2, 3, 1024, 190
    rng = np.random.default_rng(21)
    h = rng.standard_normal(N).astype(np.float32)
    r = gpu.Resampler(h, L, M, K)
    ts = torch.cuda.Stream()
    chunk = 1 << 27
    with torch.cuda.stream(ts):
        zeros = torch.zeros(K * 2 * chunk, dtype=torch.float32, device="cuda")
        d_y = torch.empty((K, 2 * (chunk * L // M + 2)), dtype=torch.float32, device="cuda")
        total = 0
        for _ in range(33):
            nf = r.process_dev(zeros.data_ptr(), 2 * chunk, d_y.data_ptr(), d_y.shape[1], stream=ts.cuda_stream)
            assert nf == 2 * (resamp_count(total + chunk, L, M) - resamp_count(total, L, M))
            total += chunk
        assert total > 2 ** 32
        x = _cx64(rng, K, 300 * M // L + 77)
        d_x = torch.from_numpy(x.view(np.float32).copy()).cuda()
        nf = r.process_dev(d_x.data_ptr() + 8, 2 * (x.shape[1] - 1), d_y.data_ptr(), d_y.shape[1],
                           in_stride=2 * x.shape[1], stream=ts.cuda_stream)
        ts.synchronize()
        y = np.ascontiguousarray(d_y.cpu().numpy()[:, :nf]).view(np.complex64)
    want = ResampPoly(h, L, M, K, start=total).process(x[:, 1:])
    _check(y, want)


def test_one_call_whose_output_spans_more_than_2_pow_31_floats(gpu):
    import torch
    K, L, M, N = 8192, 2, 1, 6
    n = (1 << 16) + 64
    n_out = resamp_count(n, L, M)
    assert K * 2 * n_out > 2 ** 31
    rng = np.random.default_rng(5)
    h = rng.standard_normal(N).astype(np.float32)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        g = torch.Generator(device="cuda").manual_seed(17)
        d_x = torch.randn(K * 2 * n, dtype=torch.float32, device="cuda", generator=g)
        d_y = torch.empty((K, 2 * n_out), dtype=torch.float32, device="cuda")
        nf = gpu.Resampler(h, L, M, K).process_dev(d_x.data_ptr(), 2 * n, d_y.data_ptr(), 2 * n_out, stream=ts.cuda_stream)
        ts.synchronize()
        assert nf == 2 * n_out
        pts = [(K - 1, n_out - 1), (0, 0), (K - 1, 0), (0, n_out - 1), (4321, n_out // 2)]
        pts += [(int(rng.integers(0, K)), int(rng.integers(0, n_out))) for _ in range(59)]
        got, want = [], []
        hT = ResampPoly(h, L, M).hT
        for k, m in pts:
            nm, phi = m * M // L, m * M % L
            row = d_x[k * 2 * n: (k + 1) * 2 * n]
            acc = 0j
            for q in range(hT.shape[1]):
                if nm - q >= 0:
                    v = row[2 * (nm - q): 2 * (nm - q) + 2].cpu().numpy()
                    acc += hT[phi, q] * complex(float(v[0]), float(v[1]))
            want.append(acc)
            got.append(complex(*d_y[k, 2 * m: 2 * m + 2].cpu().numpy()))
    got, want = np.array(got), np.array(want)
    assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()


# ---- transmit and receive -------------------------------------------------------------------------------------------
def test_transmit_at_a_dac_rate_the_symbol_rate_does_not_divide(gpu, orc):
    """QPSKModulator(4000, 1000) resampled by 5/8 to 2500 S/s (2.5 samples per symbol) matches the restatement on the
    oracle modulator's burst; resampled back by 8/5, every payload decodes at 4000 S/s."""
    rng = np.random.default_rng(8)
    h58, h85 = resamp_taps(5, 8).astype(np.float32), resamp_taps(8, 5).astype(np.float32)
    gmod = gpu.QPSKModulator(4000, SCENE_RS, 0.35, 10, tsc=TSC)
    omod = orc.QPSKModulator(4000, SCENE_RS, 0.35, 10, True, TSC)
    for _ in range(3):
        pay = rng.integers(0, 256, 48, dtype=np.uint8).tobytes()
        start = rng.integers(0, 256, 250, dtype=np.uint8).tobytes() + b"START"      # lead-in before START
        g = gmod.ModulateBytes(pay, start, b"END")
        o = omod.ModulateBytes(pay, start, b"END")
        # two leading zero samples: the round trip delays the burst by about 31 samples, and at 3 mod 4 the
        # demodulator's burst-start acquisition loses it (see resamp_oracle.resamp_scene); 33 decodes
        lead, pad = np.zeros(2 * 2, np.float32), np.zeros(2 * 200, np.float32)
        gx = np.concatenate([lead, g, pad]).view(np.complex64)
        ox = np.concatenate([lead, o, pad]).view(np.complex64)
        tx = gpu.Resampler(h58, 5, 8).process(gx)
        _check(tx, ResampPoly(h58, 5, 8).process(ox)[0])
        back = gpu.Resampler(h85, 8, 5).process(tx)
        dem = gpu.QPSKDeModulator(4000, SCENE_RS, 0.35, 10, tsc=TSC)
        assert dem.DeModulateBytes(np.ascontiguousarray(back).view(np.float32), b"START", b"END") == pay


def _receive(gpu, wide, use_fll, fse, resample=True):
    """DdcBank -> (Resampler ->) QPSKDeModulator(channels=K).demod_bytes_dev, one user stream, device calls only."""
    import torch
    K = len(SCENE_FREQS)
    bank = gpu.DdcBank(scene_taps(), SCENE_FREQS, SCENE_D)
    fs = 4000 if resample else SCENE_FS
    dem = gpu.QPSKDeModulator(fs, SCENE_RS, 0.35, 10, tsc=TSC, use_fll=use_fll, channels=K)
    if fse:
        dem.set_fractional_equalizer(21, 0.005)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        d_x = torch.from_numpy(wide.astype(np.complex64).view(np.float32).copy()).cuda()
        n_dd = wide.size // SCENE_D
        s1 = 2 * n_dd + 64
        d_dd = torch.zeros((K, s1), dtype=torch.float32, device="cuda")
        nf = bank.process_dev(d_x.data_ptr(), d_x.numel(), d_dd.data_ptr(), s1, ts.cuda_stream)
        rows, stride = d_dd, s1
        if resample:
            r = gpu.Resampler(resamp_taps(SCENE_L, SCENE_M).astype(np.float32), SCENE_L, SCENE_M, K)
            s2 = 2 * resamp_count(nf // 2, SCENE_L, SCENE_M) + 32
            d_rs = torch.zeros((K, s2), dtype=torch.float32, device="cuda")
            nf = r.process_dev(d_dd.data_ptr(), nf, d_rs.data_ptr(), s2, in_stride=s1, stream=ts.cuda_stream)
            rows, stride = d_rs, s2
        cap = 256
        d_pay = torch.zeros((K, cap), dtype=torch.uint8, device="cuda")
        d_n = torch.zeros(K, dtype=torch.int64, device="cuda")
        dem.demod_bytes_dev(rows.data_ptr(), nf, stride, b"START", b"END", d_pay.data_ptr(), cap, d_n.data_ptr(),
                            ts.cuda_stream)
        ts.synchronize()
        pay, nb = d_pay.cpu().numpy(), d_n.cpu().numpy()
        dd = np.ascontiguousarray(d_dd.cpu().numpy()[:, : 2 * n_dd]).view(np.complex64)
        out = np.ascontiguousarray(rows.cpu().numpy()[:, :nf]).view(np.complex64)
    return [pay[k, : nb[k]].tobytes() for k in range(K)], dd, out


@pytest.mark.parametrize("use_fll,fse", [(False, False), (True, False), (True, True), (False, True)])
def test_receive_chain_at_4_096_samples_per_symbol(gpu, orc, use_fll, fse):
    wide, pays = resamp_scene(orc, TSC, seed=3)
    got, dd, rs = _receive(gpu, wide, use_fll, fse)
    assert got == pays
    h = resamp_taps(SCENE_L, SCENE_M).astype(np.float32)
    _check(rs, ResampPoly(h, SCENE_L, SCENE_M, len(SCENE_FREQS)).process(dd))


def test_same_scene_without_the_resampler(gpu, orc):
    """What the chain gives at the DDC's own 4.096 samples per symbol: the fractionally spaced equalizer refuses the rate,
    and with the FLL on (designed for fs / rs = 4 by integer division) this scene's frames still decode, 4 of 4 — the
    resampler is what reaches the equalizer, not what makes the plain demodulator decode."""
    dem = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, channels=len(SCENE_FREQS))
    with pytest.raises(gpu.QpskCudaError, match="status -7"):
        dem.set_fractional_equalizer(21, 0.005)
    wide, pays = resamp_scene(orc, TSC, seed=3)
    got, _, _ = _receive(gpu, wide, use_fll=True, fse=False, resample=False)
    assert sum(g == p for g, p in zip(got, pays)) == 4
