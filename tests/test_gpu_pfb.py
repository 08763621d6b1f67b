"""GPU: the polyphase analysis channelizer (csrc/pfb.cu) against the fp64 polyphase restatement (tests/pfb_oracle.py)
within 1e-5 max|y|; bit-identical outputs for any chunking, for the host and device entry points and after reset();
untouched guard bands; argument checks; and wideband QPSK scenes demodulated straight from the channelizer's output rows."""
import ctypes as C

import numpy as np
import pytest

import kernel_variants as kv
from pfb_oracle import SCENE_FS, SCENE_RS, TSC, PfbPoly, qpsk_fdm_scene, scene_channels

pytestmark = pytest.mark.gpu


def _cx64(rng, n):
    return (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)


def _tile_blocks(M):
    """Output blocks per CTA tile of pfb_kernel (csrc/pfb.cu, pfb_run_blocks): 8192/M at every M."""
    return 8192 // M


def _check(got, want):
    assert got.shape == want.shape, (got.shape, want.shape)
    assert np.abs(got.astype(np.complex128) - want).max() <= 1e-5 * np.abs(want).max()


# the M x P grid, plus every pfb_kernel<P> at M = 4 and at M = 1024, whose tiles differ in shape (tests/kernel_variants.py)
@pytest.mark.parametrize("P,M", kv.PFB_ROWS, ids=[f"{P}-{M}" for P, M in kv.PFB_ROWS])
def test_matches_polyphase_oracle(gpu, M, P):
    rng = np.random.default_rng(M * 100 + P)
    n_taps = kv.pfb_taps(P, M)                                  # not a multiple of M (pads to P taps per branch)
    h = rng.standard_normal(n_taps) / np.sqrt(n_taps)
    n = max(40, 2 * _tile_blocks(M) + 3) * M + M // 2 + 1       # more than two tiles for every M, ragged end
    x = _cx64(rng, n)
    got = gpu.PfbChannelizer(h, M).process(x)
    want = PfbPoly(h.astype(np.float32), M).process(x)
    _check(got, want)


def test_launches_the_predicted_kernels(gpu):
    import os
    assert kv.launched_in_child("pfb", int(os.environ.get("LOCAL_RANK", "0"))) == kv.predicted_launches("pfb")


@pytest.mark.parametrize("M,P", [(4, 3), (16, 8), (64, 5), (1024, 2)])
def test_any_chunking_host_and_device_paths_and_reset_are_bit_identical(gpu, M, P):
    import torch
    rng = np.random.default_rng(7 + M)
    h = rng.standard_normal(P * M - 1)
    x = _cx64(rng, 37 * M + 5)
    one = gpu.PfbChannelizer(h, M)
    ref = one.process(x)
    _check(ref, PfbPoly(h.astype(np.float32), M).process(x))
    one.reset()
    assert np.array_equal(one.process(x).view(np.uint32), ref.view(np.uint32))
    # random chunks: odd sizes, sizes below M, empty calls
    ch = gpu.PfbChannelizer(h, M)
    cuts, a = [], 0
    while a < x.size:
        c = int(rng.choice([0, 1, 3, M - 1, M + 1, 2 * M + 7, int(rng.integers(0, 5 * M))]))
        cuts.append(min(c, x.size - a))
        a += cuts[-1]
    parts = [ch.process(x[b:b + c]) for b, c in zip(np.cumsum([0] + cuts[:-1]), cuts)]
    got = np.concatenate(parts, axis=1)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    # device path, odd float offsets into one buffer (8-byte but not 16-byte aligned blocks), same chunks.  Everything on
    # one user stream: a NULL stream would run the calls on the handle's own stream, unordered with torch's fill.
    dv = gpu.PfbChannelizer(h, M)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        d_x = torch.from_numpy(x.view(np.float32).copy()).cuda()
        stride = 2 * (x.size // M + 4)
        d_y = torch.full((M, stride), 7.0, dtype=torch.float32, device="cuda")
        col = 0
        for b, c in zip(np.cumsum([0] + cuts[:-1]), cuts):
            nf = dv.process_dev(d_x.data_ptr() + 8 * int(b), 2 * c, d_y.data_ptr() + 4 * col, stride, ts.cuda_stream)
            col += nf
        ts.synchronize()
        y = d_y.cpu().numpy()
    assert col == 2 * ref.shape[1]
    assert np.array_equal(np.ascontiguousarray(y[:, :col]).view(np.complex64).view(np.uint32), ref.view(np.uint32))
    assert np.all(y[:, col:] == 7.0)


def test_guard_bands_and_row_padding_untouched_and_repeatable(gpu):
    import torch
    M, P = 64, 8
    rng = np.random.default_rng(11)
    h = gpu.pfb_taps(M, P, 0.5 / M, 60.0)
    x = _cx64(rng, 300 * M + 17)
    n_out = x.size // M
    stride = 2 * n_out + 6
    guard = 4096
    ts = torch.cuda.Stream()
    outs = []
    for _ in range(2):
        with torch.cuda.stream(ts):
            d_x = torch.from_numpy(x.view(np.float32).copy()).cuda()
            buf = torch.full((guard + M * stride + guard,), -3.5, dtype=torch.float32, device="cuda")
            p = gpu.PfbChannelizer(h, M)
            nf = p.process_dev(d_x.data_ptr(), 2 * x.size, buf.data_ptr() + 4 * guard, stride, ts.cuda_stream)
            ts.synchronize()
            b = buf.cpu().numpy()
        assert nf == 2 * n_out
        assert np.all(b[:guard] == -3.5) and np.all(b[guard + M * stride:] == -3.5)
        rows = b[guard:guard + M * stride].reshape(M, stride)
        assert np.all(rows[:, nf:] == -3.5)
        outs.append(rows[:, :nf].copy())
    assert np.array_equal(outs[0].view(np.uint32), outs[1].view(np.uint32))
    _check(np.ascontiguousarray(outs[0]).view(np.complex64), PfbPoly(h.astype(np.float32), M).process(x))


def test_argument_checks(gpu):
    L = gpu._native.lib()
    N = gpu._native
    h = np.ones(64, np.float32) / 64
    hp = h.ctypes.data_as(N.f32p)
    out = C.c_void_p()
    assert L.qpsk_pfb_create(hp, 64, 12, C.byref(out)) == N.ERR_UNSUPPORTED
    assert L.qpsk_pfb_create(hp, 64, 2048, C.byref(out)) == N.ERR_UNSUPPORTED
    assert L.qpsk_pfb_create(hp, 64, 1, C.byref(out)) == N.ERR_UNSUPPORTED
    big = np.ones(33 * 2, np.float32)
    assert L.qpsk_pfb_create(big.ctypes.data_as(N.f32p), big.size, 2, C.byref(out)) == N.ERR_UNSUPPORTED   # P = 33
    assert L.qpsk_pfb_create(hp, 0, 16, C.byref(out)) == N.ERR_ARG
    bad = h.copy()
    bad[5] = np.inf
    assert L.qpsk_pfb_create(bad.ctypes.data_as(N.f32p), 64, 16, C.byref(out)) == N.ERR_RANGE
    bad[5] = np.nan
    assert L.qpsk_pfb_create(bad.ctypes.data_as(N.f32p), 64, 16, C.byref(out)) == N.ERR_RANGE
    with pytest.raises(gpu.ArgumentNullException):
        gpu.PfbChannelizer(None, 16)
    # odd n_floats -> ARG; a too-small stride -> CAPACITY with the needed size, and nothing consumed
    M = 16
    rng = np.random.default_rng(3)
    hh = rng.standard_normal(5 * M)
    x = _cx64(rng, 40 * M + 3)
    xf = x.view(np.float32)
    p = gpu.PfbChannelizer(hh, M)
    want = gpu.PfbChannelizer(hh, M).process(x)
    n = C.c_int64(0)
    y = np.zeros((M, 200), np.float32)
    assert L.qpsk_pfb_process(p._h, xf.ctypes.data, 7, y.ctypes.data, 200, C.byref(n)) == N.ERR_ARG
    a = 11 * M + 5                                              # first call leaves 5 samples pending
    first = p.process(x[:a])
    assert L.qpsk_pfb_process(p._h, xf[2 * a:].ctypes.data, 2 * (x.size - a), y.ctypes.data, 2, C.byref(n)) == N.ERR_CAPACITY
    assert n.value == 2 * ((x.size - a + 5) // M)
    rest = p.process(x[a:])
    got = np.concatenate([first, rest], axis=1)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert L.qpsk_pfb_process_dev(p._h, 0, 3, 0, 64, C.byref(n), None) == N.ERR_ARG


def _scene_through_device(gpu, orc, M, n_occ, seed):
    import torch
    h = gpu.pfb_taps(M, 8, 0.5 / M, 60.0)
    occ = scene_channels(M, n_occ)
    wide, pays = qpsk_fdm_scene(orc, h, M, occ, seed=seed)
    pfb = gpu.PfbChannelizer(h, M)
    dem = gpu.QPSKDeModulator(SCENE_FS, SCENE_RS, 0.35, 10, tsc=TSC, channels=M)
    # one user stream orders the buffer fills, the channelizer and the demodulator (a NULL stream would put each call on
    # its handle's own stream, with nothing ordering the demodulator's reads after the channelizer's writes)
    ts = torch.cuda.Stream()
    with torch.cuda.stream(ts):
        d_x = torch.from_numpy(wide.astype(np.complex64).view(np.float32).copy()).cuda()
        n_out = wide.size // M
        stride = 2 * n_out + 64                                 # padded rows: the demodulator reads them with in_stride
        d_y = torch.zeros((M, stride), dtype=torch.float32, device="cuda")
        cap = 256
        d_pay = torch.zeros((M, cap), dtype=torch.uint8, device="cuda")
        d_n = torch.zeros(M, dtype=torch.int64, device="cuda")
        nf = pfb.process_dev(d_x.data_ptr(), d_x.numel(), d_y.data_ptr(), stride, ts.cuda_stream)
        assert nf == 2 * n_out
        dem.demod_bytes_dev(d_y.data_ptr(), nf, stride, b"START", b"END", d_pay.data_ptr(), cap, d_n.data_ptr(), ts.cuda_stream)
        ts.synchronize()
        pay, nb, rows = d_pay.cpu().numpy(), d_n.cpu().numpy(), d_y.cpu().numpy()[:, :nf]
    return [pay[k, : nb[k]].tobytes() for k in range(M)], pays, h, wide, rows


def test_channelizer_feeds_the_batch_demodulator_4_of_16(gpu, orc):
    M = 16
    got, pays, h, wide, rows = _scene_through_device(gpu, orc, M, 4, seed=5)
    for k in range(M):
        assert got[k] == pays.get(k, b""), k
    _check(np.ascontiguousarray(rows).view(np.complex64), PfbPoly(h.astype(np.float32), M).process(wide.astype(np.complex64)))


def test_channelizer_feeds_the_batch_demodulator_64_of_256(gpu, orc):
    M = 256
    got, pays, *_ = _scene_through_device(gpu, orc, M, 64, seed=9)
    assert len(pays) == 64
    for k in range(M):
        assert got[k] == pays.get(k, b""), k
