"""GPU: the fractionally spaced form of the blind CMA equalizer (csrc/eq.cu, update stride sps) and the demodulator's
fractionally spaced stage, bit for bit against the CPU restatements in tests/fse_oracle.py (spec in include/qpskcuda.h),
plus guard-band and repeatability checks in the style of test_gpu_guards.py."""
import ctypes as C_

import numpy as np
import pytest

from fse_oracle import FseBatch, FseDemod
from test_gpu_equalizer import BENCH_CHANNEL, _bursts
from test_gpu_guards import Guarded
from test_oracle_equalizer import ALPHA, FROZEN, FROZEN_EQ, FS, RS, SPAN, TSC
from test_oracle_fse import FROZEN_FSE

pytestmark = pytest.mark.gpu

U32 = np.uint32


def _rows(orc, C, L, seed):
    return np.stack([orc.fill_uniform(seed, c, 0, 2 * L) * np.float32(1.3) for c in range(C)]).astype(np.float32)


# ---- the block ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sps", [2, 4, 3, 8])
@pytest.mark.parametrize("n_taps", [1, 7, 21, 64])
@pytest.mark.parametrize("channels", [1, 5, 64, 2048])
def test_block_matches_oracle(gpu, orc, sps, n_taps, channels):
    L = 151 if channels == 2048 else 701                 # odd: the call ends in the middle of a symbol
    x = _rows(orc, channels, L, n_taps)
    mu, modulus = 0.01, 1.2
    e = gpu.CmaEqualizer(n_taps, mu, modulus, channels=channels, sps=sps)
    got = e.Process(x if channels > 1 else x[0]).reshape(channels, -1)
    ob = FseBatch(n_taps, mu, modulus, channels, sps=sps)
    want = ob.process(x)
    for c in range(channels):
        assert np.array_equal(got[c].view(U32), want[c].view(U32)), c
    assert np.array_equal(e.taps.reshape(channels, -1).view(U32), ob.taps.view(U32))
    # the phase carried into the next call: one more block continues the stream of both
    x2 = _rows(orc, channels, 37, 3)
    got2 = e.Process(x2 if channels > 1 else x2[0]).reshape(channels, -1)
    want2 = ob.process(x2)
    for c in range(channels):
        assert np.array_equal(got2[c].view(U32), want2[c].view(U32)), c


@pytest.mark.parametrize("sps", [2, 4, 3])
@pytest.mark.parametrize("n_taps", [5, 21, 40])
def test_block_ragged_strided_and_chunked(gpu, orc, sps, n_taps):
    """Ragged counts leave the channels of a warp at different phases; the next call must carry each one's own."""
    import torch
    C, L, ld_in, ld_out = 37, 500, 523, 517
    x = _rows(orc, C, L, 100 + n_taps)
    rng = np.random.default_rng(n_taps + sps)
    n = rng.integers(0, L + 1, C).astype(np.int32)
    n[0], n[1], n[2], n[3] = L, 0, 1, 3
    mu = 0.02
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    d_in = torch.zeros((C, 2 * ld_in), dtype=torch.float32, device="cuda")
    d_in[:, : 2 * L] = torch.from_numpy(x).cuda()
    d_out = torch.full((C, 2 * ld_out), float("nan"), dtype=torch.float32, device="cuda")
    d_n = torch.from_numpy(n).cuda()
    e = gpu.CmaEqualizer(n_taps, mu, channels=C, sps=sps)
    e.process_dev(d_in.data_ptr(), d_out.data_ptr(), 2 * L, 2 * ld_in, 2 * ld_out, d_n.data_ptr(), s)
    torch.cuda.synchronize()
    got = d_out.cpu().numpy()
    ob = FseBatch(n_taps, mu, channels=C, sps=sps)
    want = ob.process(x, n)
    for c in range(C):
        k = 2 * int(n[c])
        assert np.array_equal(got[c, :k].view(U32), want[c].view(U32)), c
        assert np.isnan(got[c, k:]).all(), c                              # nothing written past the channel's count
    x2 = _rows(orc, C, 61, 7)
    got2 = e.Process(x2)
    want2 = ob.process(x2)
    for c in range(C):
        assert np.array_equal(got2[c].view(U32), want2[c].view(U32)), c
    # chunking at odd cut points (in the middle of a symbol) gives the outputs of the one-shot call
    one = gpu.CmaEqualizer(n_taps, mu, channels=C, sps=sps).Process(x)
    ch = gpu.CmaEqualizer(n_taps, mu, channels=C, sps=sps)
    cuts = [0, 2, 2 * 9, 2 * 10, 2 * 333, 2 * L]
    parts = np.concatenate([ch.Process(np.ascontiguousarray(x[:, a:b])) for a, b in zip(cuts[:-1], cuts[1:])], axis=1)
    assert np.array_equal(parts.view(U32), one.view(U32))


def test_block_reset_and_arguments(gpu, orc):
    N, C, mu = 7, 3, 0.05
    e = gpu.CmaEqualizer(N, mu, channels=C, sps=2)
    x = _rows(orc, C, 301, 3)                             # odd: the phase is 1 after the call
    y0 = e.Process(x)
    e.reset()                                             # taps, window and the sample counter
    assert np.array_equal(e.Process(x).view(U32), y0.view(U32))
    t = np.stack([orc.fill_uniform(9, c, 0, 2 * N) for c in range(C)]).astype(np.float32)
    e.taps = t
    assert np.array_equal(e.taps.view(U32), t.view(U32))
    got = e.Process(x)
    o = FseBatch(N, mu, 1.0, C, sps=2)
    o.process(x)
    o.taps = t                                            # same taps, window and phase as the handle
    want = o.process(x)
    for c in range(C):
        assert np.array_equal(got[c].view(U32), want[c].view(U32)), c
    for sps in (0, 9, -1):
        with pytest.raises(gpu.QpskCudaError, match="status -7"):
            gpu.CmaEqualizer(N, mu, sps=sps)
    with pytest.raises(gpu.ArgumentOutOfRangeException):
        gpu.CmaEqualizer(N, -1.0, sps=2)
    h = C_.c_void_p()
    assert gpu._native.lib().qpsk_eq_create_fractional(5, 0.1, 1.0, 2, 0, C_.byref(h)) == gpu._native.ERR_RANGE
    assert gpu._native.lib().qpsk_eq_create_fractional(5, 0.1, 1.0, 2, 1, None) == gpu._native.ERR_NULL


# ---- the demodulator stage ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("stages", ["fse", "fse+eq"])
@pytest.mark.parametrize("use_fll", [False, True])
def test_demod_frozen_channel_matches_oracle(gpu, orc, stages, use_fll):
    """Bits, payloads and constellation at 256 channels of the frozen channel, bit for bit with FseDemod."""
    Cn, seed = 256, 5
    bursts, _ = _bursts(gpu, orc, Cn, seed, FROZEN, 4)
    kw = dict(tsc=TSC, use_fll=use_fll)
    gd = {k: gpu.QPSKDeModulator(FS, RS, RrcAlpha=ALPHA, rrcSpan=SPAN, channels=Cn, **kw) for k in ("bits", "bytes", "cons")}
    od = {k: FseDemod(orc, FS, RS, ALPHA, SPAN, channels=Cn, **kw) for k in gd}
    for d in list(gd.values()) + list(od.values()):
        d.set_fractional_equalizer(FROZEN_FSE["n_taps"], FROZEN_FSE["mu"])
        if stages == "fse+eq":
            d.set_equalizer(FROZEN_EQ["n_taps"], FROZEN_EQ["mu"])
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
    assert frames > Cn // 2                 # frames come through (with the FLL on, the first bursts go to acquisition)
    assert np.array_equal(gd["bits"].fractional_equalizer_taps().view(U32), od["bits"].fractional_equalizer_taps().view(U32))


@pytest.mark.parametrize("use_fll", [False, True])
def test_demod_bench_geometry_matches_oracle(gpu, orc, use_fll):
    Cn, seed = 256, 11
    bursts, _ = _bursts(gpu, orc, Cn, seed, BENCH_CHANNEL, 3)
    g = gpu.QPSKDeModulator(FS, RS, RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC, use_fll=use_fll, channels=Cn)
    o = FseDemod(orc, FS, RS, ALPHA, SPAN, channels=Cn, tsc=TSC, use_fll=use_fll)
    for d in (g, o):
        d.set_fractional_equalizer(21, 0.005)
    for b, rx in enumerate(bursts):
        rx = np.ascontiguousarray(rx[:, : rx.shape[1] - 2 * 7])          # calls that do not end on a symbol boundary
        got, want = g.DeModulate(rx), o.DeModulate(rx)
        for c in range(Cn):
            assert got[c] == want[c], (b, c)


def test_identity_stage_keeps_the_bits_of_the_fused_path(gpu, orc):
    """One tap, mu 0: w = 1 and no delay, so the unfused MF -> FSE -> MM -> decode path must give the bits of the fused
    symbol-stage kernel that a handle without the stage runs."""
    Cn = 256
    bursts, _ = _bursts(gpu, orc, Cn, 17, BENCH_CHANNEL, 3)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC)
    a = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    b = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    b.set_fractional_equalizer(1, 0.0)
    for rx in bursts:
        assert a.DeModulate(rx) == b.DeModulate(rx)
    b.set_fractional_equalizer(0, 0.0)                    # off again: back on the fused path, loop state intact
    assert a.DeModulate(bursts[0]) == b.DeModulate(bursts[0])
    with pytest.raises(gpu.ArgumentException):
        b.fractional_equalizer_taps()


def test_set_fractional_equalizer_arguments_and_independence(gpu, orc):
    Cn = 4
    bursts, _ = _bursts(gpu, orc, Cn, 23, FROZEN, 4)
    kw = dict(RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC)
    a = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    b = gpu.QPSKDeModulator(FS, RS, channels=Cn, **kw)
    for d in (a, b):
        d.set_fractional_equalizer(21, 0.005)
        d.set_equalizer(11, 0.01)
    assert a.DeModulate(bursts[0]) == b.DeModulate(bursts[0])
    # refused calls consume no state
    for args in [(21, -0.1), (21, 0.01, 0.0), (21, float("nan"))]:
        with pytest.raises(gpu.ArgumentOutOfRangeException):
            b.set_fractional_equalizer(*args)
    for n in (65, -1):
        with pytest.raises(gpu.QpskCudaError, match="status -7"):
            b.set_fractional_equalizer(n, 0.01)
    assert a.DeModulate(bursts[1]) == b.DeModulate(bursts[1])
    assert np.array_equal(a.fractional_equalizer_taps().view(U32), b.fractional_equalizer_taps().view(U32))
    # setting one stage resets that stage only: as the oracle doing the same at the same point
    o = FseDemod(orc, FS, RS, ALPHA, SPAN, channels=Cn, tsc=TSC)
    o.set_fractional_equalizer(21, 0.005)
    o.set_equalizer(11, 0.01)
    o.DeModulate(bursts[0])
    o.DeModulate(bursts[1])
    o.set_fractional_equalizer(15, 0.01)
    a.set_fractional_equalizer(15, 0.01)
    assert a.DeModulate(bursts[2]) == o.DeModulate(bursts[2])
    o.set_equalizer(7, 0.02)
    a.set_equalizer(7, 0.02)
    assert a.DeModulate(bursts[3]) == o.DeModulate(bursts[3])
    assert np.array_equal(a.fractional_equalizer_taps().view(U32), o.fractional_equalizer_taps().view(U32))
    assert np.array_equal(a.equalizer_taps().view(U32), o.equalizer_taps().view(U32))
    # the stage needs an integer rate of 2..8 samples per symbol; turning it off is always accepted
    for fs, rs in ((10_000_000, 3_000_000), (5_000_000, 5_000_000), (9_000_000, 1_000_000)):
        d = gpu.QPSKDeModulator(fs, rs, RrcAlpha=ALPHA, rrcSpan=SPAN)
        with pytest.raises(gpu.QpskCudaError, match="status -7"):
            d.set_fractional_equalizer(11, 0.01)
        d.set_fractional_equalizer(0, 0.0)


def test_streaming_demodulator_with_fractional_equalizer(gpu, orc):
    bursts, _ = _bursts(gpu, orc, 1, 29, FROZEN, 8)
    blocks = [r[0] for r in bursts]
    od = FseDemod(orc, FS, RS, ALPHA, SPAN, tsc=TSC)
    od.set_fractional_equalizer(FROZEN_FSE["n_taps"], FROZEN_FSE["mu"])
    want = [od.DeModulateBytes(b[None, :], b"S", b"E")[0] for b in blocks]
    per_call = gpu.QPSKDeModulator(FS, RS, RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC)
    per_call.set_fractional_equalizer(FROZEN_FSE["n_taps"], FROZEN_FSE["mu"])
    assert [per_call.DeModulateBytes(b, b"S", b"E") for b in blocks] == want
    gd = gpu.QPSKDeModulator(FS, RS, RrcAlpha=ALPHA, rrcSpan=SPAN, tsc=TSC)
    gd.set_fractional_equalizer(FROZEN_FSE["n_taps"], FROZEN_FSE["mu"])
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
    assert sum(len(p) > 0 for p in want) >= 2


# ---- guard bands ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sps", [2, 4, 3])
def test_block_dev_outputs_stay_in_bounds_and_repeat(gpu, sps):
    import torch
    for C, L, n_taps in ((1, 257, 21), (5, 1000, 64), (37, 333, 11), (2049, 65, 31)):
        ld = 2 * L + 2
        x = torch.empty(C * ld, dtype=torch.float32, device="cuda")
        gpu.fill_uniform_dev(6, 0, 0, x.numel(), x.data_ptr(), 0)
        torch.cuda.synchronize()
        outs = []
        for rep in range(3):
            g = Guarded(torch, C * ld * 4)
            e = gpu.CmaEqualizer(n_taps, 0.01, channels=C, sps=sps)
            e.process_dev(x.data_ptr(), g.ptr, 2 * L, ld, ld)
            e.process_dev(x.data_ptr(), g.ptr, 2 * L, ld, ld)                 # a second call on the carried state
            torch.cuda.synchronize()
            g.check(f"fse sps={sps} C={C}")
            y = g.f32().view(C, ld)
            assert bool((y[:, 2 * L:].contiguous().view(torch.uint8) == 0xA5).all())
            outs.append(y[:, : 2 * L].clone())
            e.close()
        assert all(torch.equal(outs[0], o) for o in outs[1:]), (C, L)


@pytest.mark.parametrize("use_fll", [False, True])
def test_demod_dev_with_stage_stays_in_bounds_and_repeats(gpu, use_fll):
    import torch
    alpha = float(np.float32(0.4))
    for C, n_payload in ((1, 40), (33, 200), (70, 600)):
        mod = gpu.QPSKModulator(FS, RS, alpha, 10, True, TSC)
        pay = torch.empty((C, n_payload), dtype=torch.uint8, device="cuda")
        gpu.fill_bytes_dev(4, 0, C, n_payload, pay.data_ptr(), 0)
        ff = mod.frame_floats(n_payload, b"S", b"E")
        tx = torch.empty((C, ff), dtype=torch.float32, device="cuda")
        mod.modulate_frames_dev(pay.data_ptr(), n_payload, C, b"S", b"E", tx.data_ptr(), ff)
        rx = torch.empty_like(tx)
        ch = gpu.SimChannel(100e6, 100e6, FS, 1, 1, noise_dbfs=-40.0, mode=1, path_gains_iq=(1.0, 0.0, 0.12, 0.08), path_delays=(0, 3),
                            seed=9, channels=C, first_channel=0)
        ch.apply_dev(tx.data_ptr(), ff, ff, rx.data_ptr(), ff)
        torch.cuda.synchronize()
        runs = []
        for rep in range(3):
            dem = gpu.QPSKDeModulator(FS, RS, alpha, 10, tsc=TSC, use_fll=use_fll, channels=C, max_frame_bytes=2048)
            dem.set_fractional_equalizer(21, 0.005)
            cap = dem.bits_bound(ff)
            gb = Guarded(torch, C * cap)
            gn = Guarded(torch, C * 8)
            gp = Guarded(torch, C * 1024)
            gnp = Guarded(torch, C * 8)
            dem.demod_bits_dev(rx.data_ptr(), ff, ff, gb.ptr, cap, gn.ptr)
            dem2 = gpu.QPSKDeModulator(FS, RS, alpha, 10, tsc=TSC, use_fll=use_fll, channels=C, max_frame_bytes=2048)
            dem2.set_fractional_equalizer(21, 0.005)
            dem2.demod_bytes_dev(rx.data_ptr(), ff, ff, b"S", b"E", gp.ptr, 1024, gnp.ptr)
            torch.cuda.synchronize()
            for g, w in ((gb, "bits"), (gn, "bit counts"), (gp, "payload"), (gnp, "payload lengths")):
                g.check(f"demod+fse {w} C={C} fll={use_fll}")
            nb = gn.body().view(torch.int64).clone()
            bits = gb.body().view(C, cap)
            for c in range(C):
                assert bool((bits[c, int(nb[c]):] == 0xA5).all()) or int(nb[c]) == 0, (C, c)
            runs.append((nb, torch.stack([bits[c, : int(nb.min())] for c in range(C)]).clone(), gnp.body().clone()))
        for r in runs[1:]:
            assert torch.equal(runs[0][0], r[0]) and torch.equal(runs[0][1], r[1]) and torch.equal(runs[0][2], r[2])
