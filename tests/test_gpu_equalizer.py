"""GPU: the blind CMA equalizer block (csrc/eq.cu) and the demodulator's opt-in equalizer stage, bit for bit against the
CPU restatements in tests/cma_oracle.py (spec in include/qpskcuda.h)."""
import numpy as np
import pytest

from cma_oracle import CmaBatch, EqDemod
from test_oracle_equalizer import (ALPHA, BURSTS, FROZEN, FROZEN_EQ, FS, RS, SPAN, TSC, burst_errors, frozen_frame)

pytestmark = pytest.mark.gpu

U32 = np.uint32


def _rows(orc, C, L, seed):
    return np.stack([orc.fill_uniform(seed, c, 0, 2 * L) * np.float32(1.3) for c in range(C)]).astype(np.float32)


def _oracle_rows(x, n_taps, mu, modulus=1.0, lengths=None):
    b = CmaBatch(n_taps, mu, modulus, x.shape[0])
    return b.process(x, lengths), b


@pytest.mark.parametrize("n_taps", [1, 2, 7, 11, 33, 64])
@pytest.mark.parametrize("channels", [1, 5, 64, 2048])
def test_block_matches_oracle(gpu, orc, n_taps, channels):
    L = 150 if channels == 2048 else 700
    x = _rows(orc, channels, L, n_taps)
    mu, modulus = 0.01, 1.2
    e = gpu.CmaEqualizer(n_taps, mu, modulus, channels=channels)
    got = e.Process(x if channels > 1 else x[0])
    got = got.reshape(channels, -1)
    want, ob = _oracle_rows(x, n_taps, mu, modulus)
    for c in range(channels):
        assert np.array_equal(got[c].view(U32), want[c].view(U32)), c
    assert np.array_equal(e.taps.reshape(channels, -1).view(U32), ob.taps.view(U32))


@pytest.mark.parametrize("n_taps", [5, 11, 40])
def test_block_ragged_strided_and_chunked(gpu, orc, n_taps):
    import torch
    C, L, ld_in, ld_out = 37, 500, 523, 517
    x = _rows(orc, C, L, 100 + n_taps)
    rng = np.random.default_rng(n_taps)
    n = rng.integers(0, L + 1, C).astype(np.int32)
    n[0], n[1], n[2] = L, 0, 1
    mu = 0.02
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    d_in = torch.zeros((C, 2 * ld_in), dtype=torch.float32, device="cuda")
    d_in[:, : 2 * L] = torch.from_numpy(x).cuda()
    d_out = torch.full((C, 2 * ld_out), float("nan"), dtype=torch.float32, device="cuda")
    d_n = torch.from_numpy(n).cuda()
    e = gpu.CmaEqualizer(n_taps, mu, channels=C)
    e.process_dev(d_in.data_ptr(), d_out.data_ptr(), 2 * L, 2 * ld_in, 2 * ld_out, d_n.data_ptr(), s)
    torch.cuda.synchronize()
    got = d_out.cpu().numpy()
    want, ob = _oracle_rows(x, n_taps, mu, lengths=n)
    for c in range(C):
        k = 2 * int(n[c])
        assert np.array_equal(got[c, :k].view(U32), want[c].view(U32)), c
        assert np.isnan(got[c, k:]).all(), c                              # nothing written past the channel's count
    # the state each channel carries on is that of its own n[c] symbols: continue with the rest of the rows, one-shot
    x2 = _rows(orc, C, 60, 7)
    got2 = e.Process(x2)
    want2 = ob.process(x2)
    for c in range(C):
        assert np.array_equal(got2[c].view(U32), want2[c].view(U32)), c
    # arbitrary chunking of a stream gives the bits of the one-shot call
    one = gpu.CmaEqualizer(n_taps, mu, channels=C).Process(x)
    ch = gpu.CmaEqualizer(n_taps, mu, channels=C)
    cuts = [0, 2, 2 * 9, 2 * 10, 2 * 333, 2 * L]
    parts = np.concatenate([ch.Process(np.ascontiguousarray(x[:, a:b])) for a, b in zip(cuts[:-1], cuts[1:])], axis=1)
    assert np.array_equal(parts.view(U32), one.view(U32))


def test_block_taps_reset_and_arguments(gpu, orc):
    N, C, mu = 7, 3, 0.05
    e = gpu.CmaEqualizer(N, mu, channels=C)
    spike = np.zeros((C, 2 * N), np.float32)
    spike[:, 2 * 3] = 1.0
    assert np.array_equal(e.taps, spike)
    x = _rows(orc, C, 300, 3)
    y0 = e.Process(x)
    moved = e.taps
    assert not np.array_equal(moved, spike)
    e.reset()
    assert np.array_equal(e.taps, spike)
    assert np.array_equal(e.Process(x).view(U32), y0.view(U32))
    # set / get round trip, and the outputs follow the taps that were set (oracle started from the same taps)
    t = np.stack([orc.fill_uniform(9, c, 0, 2 * N) for c in range(C)]).astype(np.float32)
    e.reset()
    e.taps = t
    assert np.array_equal(e.taps.view(U32), t.view(U32))
    # refused calls leave the state where it was
    with pytest.raises(gpu.ArgumentException):
        e.taps = t[:, :-2]
    bad = t.copy()
    bad[1, 3] = np.inf
    with pytest.raises(gpu.ArgumentOutOfRangeException):
        e.taps = bad
    with pytest.raises(gpu.ArgumentException):
        e.Process(x[:, :5])
    with pytest.raises(gpu.QpskCudaError, match="status -6"):
        e.Process(x, np.empty((C, x.shape[1] - 2), np.float32))
    import ctypes as C_
    small = np.empty(C * 2 * N - 1, np.float32)
    assert gpu._native.lib().qpsk_eq_get_taps(e._h, small.ctypes.data_as(gpu._native.f32p), small.size) == gpu._native.ERR_CAPACITY
    assert np.array_equal(e.taps.view(U32), t.view(U32))
    got = e.Process(x)
    o = CmaBatch(N, mu, 1.0, C)
    o.taps = t
    want = o.process(x)
    for c in range(C):
        assert np.array_equal(got[c].view(U32), want[c].view(U32)), c
    for args, exc in [((7, -1.0), gpu.ArgumentOutOfRangeException), ((7, float("inf")), gpu.ArgumentOutOfRangeException),
                      ((7, 0.1, 0.0), gpu.ArgumentOutOfRangeException), ((7, 0.1, float("nan")), gpu.ArgumentOutOfRangeException)]:
        with pytest.raises(exc):
            gpu.CmaEqualizer(*args)
    for n in (0, 65, -3):
        with pytest.raises(gpu.QpskCudaError, match="status -7"):
            gpu.CmaEqualizer(n, 0.1)
    h = C_.c_void_p()
    assert gpu._native.lib().qpsk_eq_create_batch(5, 0.1, 1.0, 0, C_.byref(h)) == gpu._native.ERR_RANGE


# ---------------------------------------------------------------------------------------------------------------------
# the demodulator's equalizer stage
# ---------------------------------------------------------------------------------------------------------------------
BENCH_CHANNEL = dict(path_gains_iq=(1.0, 0.0, 0.12, 0.08), path_delays=(0, 3), noise_dbfs=-40.0)


def _sim(gpu, Cn, seed, channel):
    return gpu.SimChannel(100e6, 100e6, FS, 1, 1, noise_dbfs=channel["noise_dbfs"], mode=1, path_gains_iq=channel["path_gains_iq"],
                          path_delays=channel["path_delays"], seed=seed, channels=Cn)


def _bursts(gpu, orc, Cn, seed, channel, n_bursts):
    """n_bursts consecutive blocks of the same frame through the GPU channel simulator -> host arrays [Cn, n]."""
    import torch
    tx, ref = frozen_frame(orc, seed)
    ch = _sim(gpu, Cn, seed, channel)
    d_tx = torch.from_numpy(tx).cuda()
    d_rx = torch.empty((Cn, tx.size), dtype=torch.float32, device="cuda")
    out = []
    for _ in range(n_bursts):
        ch.apply_dev(d_tx.data_ptr(), tx.size, 0, d_rx.data_ptr(), tx.size, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        out.append(d_rx.cpu().numpy())
    return out, ref


def test_demod_frozen_channel_matches_oracle_and_recovers(gpu, orc):
    Cn, seed = 256, 5
    bursts, ref = _bursts(gpu, orc, Cn, seed, FROZEN, BURSTS)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=SPAN)
    g_on = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    g_on.set_equalizer(FROZEN_EQ["n_taps"], FROZEN_EQ["mu"])
    g_off = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    o_on = EqDemod(orc, FS, RS, ALPHA, SPAN, channels=Cn)
    o_on.set_equalizer(FROZEN_EQ["n_taps"], FROZEN_EQ["mu"])
    o_off = [orc.QPSKDeModulator(FS, RS, ALPHA, SPAN) for _ in range(Cn)]
    cnt = {k: np.zeros((Cn, 2), np.int64) for k in ("gpu_on", "gpu_off", "orc_on", "orc_off")}
    for b, rx in enumerate(bursts):
        gon, goff, oon = g_on.DeModulate(rx), g_off.DeModulate(rx), o_on.DeModulate(rx)
        for c in range(Cn):
            won, woff = oon[c], o_off[c].DeModulate(rx[c])
            assert gon[c] == won and goff[c] == woff, (b, c)
            if b == 0:
                continue                                                   # acquisition
            for k, bits in (("gpu_on", gon[c]), ("gpu_off", goff[c]), ("orc_on", won), ("orc_off", woff)):
                cnt[k][c] += burst_errors(np.frombuffer(bits.encode(), np.uint8) - ord("0"), ref)
    assert np.array_equal(cnt["gpu_on"], cnt["orc_on"]) and np.array_equal(cnt["gpu_off"], cnt["orc_off"])
    ber_on = cnt["gpu_on"][:, 0].sum() / cnt["gpu_on"][:, 1].sum()
    ber_off = cnt["gpu_off"][:, 0].sum() / cnt["gpu_off"][:, 1].sum()
    assert ber_off >= 1e-2, ber_off
    # Mueller-Muller runs on the unequalized eye: on a few channels (LO drift draws) its timing slips and the burst after
    # the slip is lost, so the bound of the CPU test's channel holds for the typical channel, not for every one
    assert np.median(cnt["gpu_on"][:, 0] / cnt["gpu_on"][:, 1]) <= 1e-3, cnt["gpu_on"][:, 0]
    assert ber_on <= ber_off / 20, (ber_on, ber_off)
    taps = g_on.equalizer_taps()
    assert np.array_equal(taps.view(U32), o_on.equalizer_taps().view(U32))


@pytest.mark.parametrize("use_fll", [False, True])
@pytest.mark.parametrize("tsc", [TSC, None])
def test_demod_bench_geometry_matches_oracle(gpu, orc, use_fll, tsc):
    """sps 2, 21-tap matched filter, the benchmark's echo: bits, payloads and constellation with the stage on."""
    Cn, seed, n_b = 256, 11, 3
    bursts, _ = _bursts(gpu, orc, Cn, seed, BENCH_CHANNEL, n_b)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=tsc, use_fll=use_fll)
    gd = {k: gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw) for k in ("bits", "bytes", "cons")}
    for g in gd.values():
        g.set_equalizer(11, 0.005)
    od = {k: EqDemod(orc, FS, RS, ALPHA, SPAN, channels=Cn, tsc=tsc, use_fll=use_fll) for k in gd}
    for o in od.values():
        o.set_equalizer(11, 0.005)
    frames = 0
    for b, rx in enumerate(bursts):
        bits = gd["bits"].DeModulate(rx)
        pays = gd["bytes"].DeModulateBytes(rx, b"S", b"E")
        cons = gd["cons"].deModulateConstellation(rx)
        wbits, wpays, wcons = od["bits"].DeModulate(rx), od["bytes"].DeModulateBytes(rx, b"S", b"E"), od["cons"].deModulateConstellation(rx)
        for c in range(Cn):
            assert bits[c] == wbits[c], (b, c)
            assert pays[c] == wpays[c], (b, c)
            frames += len(wpays[c]) > 0
            assert np.array_equal(cons[c].view(U32), wcons[c].view(U32)), (b, c)
    assert frames > Cn                                                     # the stage decodes this channel


def test_identity_equalizer_keeps_the_bits_of_the_fused_path(gpu, orc):
    """One tap, mu 0: w = 1 and no delay, so the unfused MM -> EQ -> decode path must give the bits of the fused
    symbol-stage kernel that a handle without the stage runs."""
    Cn = 256
    bursts, _ = _bursts(gpu, orc, Cn, 17, BENCH_CHANNEL, 3)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC)
    a = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    b = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    b.set_equalizer(1, 0.0)
    for rx in bursts:
        assert a.DeModulate(rx) == b.DeModulate(rx)
    # turning the stage off again returns the handle to the fused path with its loop state intact
    b.set_equalizer(0, 0.0)
    assert a.DeModulate(bursts[0]) == b.DeModulate(bursts[0])
    with pytest.raises(gpu.ArgumentException):
        b.equalizer_taps()


def test_demod_set_equalizer_arguments_leave_state(gpu, orc):
    Cn = 4
    bursts, _ = _bursts(gpu, orc, Cn, 23, FROZEN, 3)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC)
    a = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    b = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    a.set_equalizer(11, 0.01)
    b.set_equalizer(11, 0.01)
    assert a.DeModulate(bursts[0]) == b.DeModulate(bursts[0])
    for args in [(11, -0.1), (11, 0.01, 0.0), (11, float("nan"))]:
        with pytest.raises(gpu.ArgumentOutOfRangeException):
            b.set_equalizer(*args)
    for n in (65, -1):
        with pytest.raises(gpu.QpskCudaError, match="status -7"):
            b.set_equalizer(n, 0.01)
    assert a.DeModulate(bursts[1]) == b.DeModulate(bursts[1])
    assert np.array_equal(a.equalizer_taps().view(U32), b.equalizer_taps().view(U32))
    # set_equalizer resets the equalizer only: the same as the oracle doing the same at the same point
    o = EqDemod(orc, FS, RS, ALPHA, SPAN, channels=Cn, tsc=TSC)
    o.set_equalizer(11, 0.01)
    o.DeModulate(bursts[0])
    o.DeModulate(bursts[1])
    o.set_equalizer(7, 0.02)
    a.set_equalizer(7, 0.02)
    assert a.DeModulate(bursts[2]) == o.DeModulate(bursts[2])


def test_streaming_demodulator_with_equalizer(gpu, orc):
    bursts, _ = _bursts(gpu, orc, 1, 29, FROZEN, 8)
    blocks = [r[0] for r in bursts]
    od = EqDemod(orc, FS, RS, ALPHA, SPAN, tsc=TSC)
    od.set_equalizer(FROZEN_EQ["n_taps"], FROZEN_EQ["mu"])
    want = [od.DeModulateBytes(b[None, :], b"S", b"E")[0] for b in blocks]
    per_call = gpu.QPSKDeModulator(FS, RS, RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC)
    per_call.set_equalizer(FROZEN_EQ["n_taps"], FROZEN_EQ["mu"])
    assert [per_call.DeModulateBytes(b, b"S", b"E") for b in blocks] == want
    gd = gpu.QPSKDeModulator(FS, RS, RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC)
    gd.set_equalizer(FROZEN_EQ["n_taps"], FROZEN_EQ["mu"])
    st = gpu.StreamingDemodulator(gd, b"S", b"E", max_block_floats=max(b.size for b in blocks), max_payload_bytes=1 << 16, depth=3)
    got = []
    for b in blocks:
        st.push(b)
        p = st.poll()
        if p is not None:
            got.append(p)
    got += st.drain()
    st.close()
    assert got == want
    assert sum(len(p) > 0 for p in want) >= 2                           # frames do come through the equalized stream
