"""GPU tests of the drop-in boundary's behaviour (round-2 review items): what the span overloads RETURN, that a refused
call leaves the stream where it was, that a frame grown over many small calls is not lost to a buffer sized from one
call, and that a handle keeps the device it was created on.  All through the C ABI (ctypes mirror), checked against the
oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"


def _burst(orc, n_payload=96, fs=4000, rs=1000, seed=3, tsc=None, sm=b"S", em=b"E"):
    rng = np.random.default_rng(seed)
    p = rng.integers(0, 256, n_payload, dtype=np.uint8).tobytes()
    return orc.QPSKModulator(fs, rs, 0.35, 10, True, tsc).ModulateBytes(p, sm, em), p


def test_span_overloads_return_the_reference_counts(gpu, orc):
    """Process(ReadOnlySpan<float>, Span<float>) returns COMPLEX samples for the FLL (Band-Edge Filter.cs:71,86) and the
    Costas loop (CostasLoopQpsk.cs:105,113) and complex SYMBOLS for Mueller-Muller (MuellerMuller.cs:135) — the count
    QPSKDeModulator.cs:364-375 loops over.  The allocating overloads return 2x that many floats."""
    x, _ = _burst(orc)
    n = x.size
    f, of = gpu.FLLBandEdgeFilter(4.0, 0.35, 40, 0.01), orc.FLLBandEdgeFilter(4.0, 0.35, 40, 0.01)
    y = np.empty(n, np.float32)
    assert f.Process(x, y) == n >> 1
    assert np.array_equal(y, of.Process(x))
    mf = orc.ComplexFIRFilter(orc.real_taps_to_iq(orc.RRCFilter.generateCoefficents(10, 0.35, 4000, 1000))).Filter(x)
    kp, ki = gpu.mm_gains_from_bw(0.002)
    m, om = gpu.MuellerMuller(4.0, kp, ki), orc.MuellerMuller(4.0, kp, ki)
    want = om.Process(mf)
    sym = np.zeros(n, np.float32)
    ns = m.Process(mf, sym)
    assert isinstance(ns, int) and ns == want.size >> 1 and 0 < ns < n >> 1
    assert np.allclose(sym[: ns << 1], want, rtol=0, atol=1e-5 * np.abs(want).max())
    m2 = gpu.MuellerMuller(4.0, kp, ki)
    assert m2.Process(mf).size == ns << 1                       # float[] overload: n << 1 floats (:154)
    c, oc = gpu.CostasLoopQpsk(1000.0, 10.0), orc.CostasLoopQpsk(1000.0, 10.0)
    out = np.empty(ns << 1, np.float32)
    assert c.Process(want, out) == ns
    wc = oc.Process(want)
    assert np.allclose(out, wc, rtol=0, atol=1e-5 * np.abs(wc).max())


def test_frame_grown_over_many_small_calls_is_not_lost(gpu, orc):
    """ADVICE r1: the framer ring persists across calls, so the call that completes a frame can return a payload far
    longer than a buffer sized from that call's own samples (the MTU-block loop of ModDemodOverSDR.cs:127-136).  The
    host call reports the size, the frame stays in the ring, and the Python / C# host fetches it — same payloads as the
    oracle, call by call."""
    fs, rs = 4000, 1000
    sm, em = b"\xa5GO", b"END\x5a"
    x, payload = _burst(orc, n_payload=1500, sm=sm, em=em)
    kw = dict(RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002)
    od, gd = orc.QPSKDeModulator(fs, rs, **kw), gpu.QPSKDeModulator(fs, rs, **kw)
    gd.set_fir_mode(gpu.FIR_EXACT)
    chunk = 2 * 64                                              # 64 samples -> ~16 symbols -> 4 payload bytes per call
    got = []
    for a in range(0, x.size, chunk):
        w = od.DeModulateBytes(x[a:a + chunk], sm, em, cap=4096)
        g = gd.DeModulateBytes(x[a:a + chunk], sm, em)          # default cap: n // 8 + 64 = 80 bytes << 1500
        assert g == w, a
        if g:
            got.append(g)
    assert got == [payload]
    # the raw C call: CAPACITY with the needed size, then qpsk_demod_last_payload returns the frame
    import ctypes as C
    L = gpu._native.lib()
    gd2 = gpu.QPSKDeModulator(fs, rs, **kw)
    gd2.set_fir_mode(gpu.FIR_EXACT)
    s, e = np.frombuffer(sm, np.uint8).copy(), np.frombuffer(em, np.uint8).copy()
    small = np.zeros(16, np.uint8)
    nb = np.zeros(1, np.int64)
    seen = None
    for a in range(0, x.size, chunk):
        xc = np.ascontiguousarray(x[a:a + chunk])
        st = L.qpsk_demod_bytes(gd2._h, xc.ctypes.data, xc.size, s.ctypes.data, s.size, e.ctypes.data, e.size, small.ctypes.data, 16,
                                nb.ctypes.data)
        if st == gpu._native.ERR_CAPACITY:
            assert nb[0] == len(payload)
            big = np.zeros(int(nb[0]), np.uint8)
            nb2 = np.zeros(1, np.int64)
            assert L.qpsk_demod_last_payload(gd2._h, big.ctypes.data, big.size, nb2.ctypes.data) == 0 and nb2[0] == nb[0]
            seen = big.tobytes()
        else:
            assert st == 0 and nb[0] == 0
    assert seen == payload
    del C


def test_refused_device_call_leaves_the_stream_untouched(gpu, orc):
    """ADVICE r1: capacity / alignment errors of the *_dev entry points are reported before any stage consumes samples:
    after a refused call the same samples still demodulate to the oracle's bits.  With an opt-in stage on (AGC W = 64,
    fractionally spaced or symbol-spaced equalizer) they demodulate to the bits of a twin handle that saw no refused call."""
    import torch
    fs, rs = 4000, 1000
    x, _ = _burst(orc, n_payload=200, tsc=None)
    kw = dict(RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002)
    L = gpu._native.lib()
    dx = torch.from_numpy(x).cuda()

    def handle(use_fll, stage):
        gd = gpu.QPSKDeModulator(fs, rs, use_fll=use_fll, **kw)
        gd.set_fir_mode(gpu.FIR_EXACT)
        if stage == "agc":
            gd.set_agc(64)
        elif stage == "fse":
            gd.set_fractional_equalizer(11, 0.01)
        elif stage == "eq":
            gd.set_equalizer(11, 0.01)
        return gd

    def bits(gd, refuse):
        cap = gd.bits_bound(x.size)
        out = torch.zeros(cap + 2, dtype=torch.uint8, device="cuda")
        nb = torch.zeros(1, dtype=torch.int64, device="cuda")
        if refuse:
            with pytest.raises(gpu.QpskCudaError):              # too small: QPSK_ERR_CAPACITY
                gd.demod_bits_dev(dx.data_ptr(), x.size, x.size, out.data_ptr(), 8, nb.data_ptr())
            with pytest.raises(gpu.ArgumentException):          # odd output address (uchar2 stores): QPSK_ERR_ARG
                gd.demod_bits_dev(dx.data_ptr(), x.size, x.size, out.data_ptr() + 1, cap, nb.data_ptr())
        gd.demod_bits_dev(dx.data_ptr(), x.size, x.size, out.data_ptr(), cap, nb.data_ptr())
        torch.cuda.synchronize()
        return "".join("1" if b else "0" for b in out[: int(nb.item())].cpu().numpy())

    def constellation(gd, refuse):
        # short output refused before the matched filter / MM advance
        sym = torch.zeros(x.size, dtype=torch.float32, device="cuda")
        ns = torch.zeros(1, dtype=torch.int32, device="cuda")
        if refuse:
            assert L.qpsk_demod_constellation_dev(gd._h, dx.data_ptr(), x.size, x.size, sym.data_ptr(), 8, ns.data_ptr(),
                                                  None) == gpu._native.ERR_CAPACITY
        assert L.qpsk_demod_constellation_dev(gd._h, dx.data_ptr(), x.size, x.size, sym.data_ptr(), x.size, ns.data_ptr(),
                                              None) == 0
        torch.cuda.synchronize()
        return sym[: 2 * int(ns.item())].cpu().numpy()

    for use_fll in (False, True):
        want = orc.QPSKDeModulator(fs, rs, use_fll=use_fll, **kw).DeModulate(x)
        assert bits(handle(use_fll, None), True) == want and len(want) > 100
        for stage in ("agc", "fse", "eq"):
            got = bits(handle(use_fll, stage), True)
            assert got == bits(handle(use_fll, stage), False) and len(got) > 100, (use_fll, stage)
    wc = orc.QPSKDeModulator(fs, rs, **kw).deModulateConstellation(x)
    got = constellation(handle(False, None), True)
    assert got.size == wc.size
    assert np.allclose(got, wc, rtol=0, atol=1e-5 * np.abs(wc).max())
    for stage in ("agc", "fse", "eq"):
        got = constellation(handle(False, stage), True)
        assert got.size > 100 and np.array_equal(got.view(np.uint32), constellation(handle(False, stage), False).view(np.uint32)), stage


def test_handles_keep_the_device_they_were_created_on(gpu, orc):
    """ADVICE r1: no handle relied on a process-global device.  Each handle records its ordinal; calls select it whatever
    qpsk_set_device says at the time, and threads choose devices independently.  With one GPU visible only the
    bookkeeping can be checked; with two, a handle created on device 0 is driven after the default moved to device 1."""
    import ctypes as C
    L = gpu._native.lib()
    gd = gpu.QPSKDeModulator(4000, 1000, RrcAlpha=0.35, rrcSpan=10)
    dev = C.c_int(-1)
    assert L.qpsk_demod_device(gd._h, C.byref(dev)) == 0 and dev.value == 0
    n = gpu.device_count()
    with pytest.raises(gpu.QpskCudaError):
        gpu.set_device(n)                                       # refused, and the previous choice stays in force
    assert gpu.ComplexFIRFilter(np.array([1, 0], np.float32)).Filter(np.ones(4, np.float32)).tolist() == [1, 1, 1, 1]
    if n < 2:
        return
    x, _ = _burst(orc)
    want = orc.QPSKDeModulator(4000, 1000, RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002).DeModulate(x)
    g0 = gpu.QPSKDeModulator(4000, 1000, RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002)
    g0.set_fir_mode(gpu.FIR_EXACT)
    try:
        gpu.set_device(1)
        g1 = gpu.QPSKDeModulator(4000, 1000, RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002)
        g1.set_fir_mode(gpu.FIR_EXACT)
        assert L.qpsk_demod_device(g1._h, C.byref(dev)) == 0 and dev.value == 1
        assert g0.DeModulate(x) == want                         # device-0 handle while the default is device 1
        assert g1.DeModulate(x) == want
    finally:
        gpu.set_device(0)


def test_counter_gather_through_the_c_abi_single_rank(gpu):
    """qpsk_comm_* / qpsk_ber_gather (csrc/comm.cu): the library's own NCCL communicator.  One GPU here, so the
    communicator has one rank (an all-gather over one rank); bench.py runs the same calls at N = 2, 4, 8."""
    import torch
    from qpsk_modulator_demodulator_b200 import shard
    comm = shard.CounterComm(1, 0, lambda ident: ident)
    info = comm.info()
    assert info["n_ranks"] == 1 and info["rank"] == 0 and info["nccl_version"] >= 21000
    C = 37
    cnt = torch.stack([torch.arange(C, dtype=torch.int32), torch.arange(C, dtype=torch.int32) + 1000], dim=1).contiguous().cuda()
    torch.cuda.synchronize()
    allc = comm.gather(cnt.data_ptr(), C, C)
    assert allc.shape == (C, 2) and np.array_equal(allc[:, 0], np.arange(C)) and np.array_equal(allc[:, 1], np.arange(C) + 1000)
    # ragged: the block is shorter than the common width -> padded rows are dropped again by the host mirror
    L = gpu._native.lib()
    out = np.zeros((1, 40, 2), np.uint32)
    assert L.qpsk_ber_gather(comm._h, cnt.data_ptr(), C, 40, out.ctypes.data) == 0
    assert np.array_equal(out[0, :C, 1], np.arange(C) + 1000) and not out[0, C:].any()
    assert L.qpsk_ber_gather(comm._h, cnt.data_ptr(), 41, 40, out.ctypes.data) == gpu._native.ERR_RANGE
    comm.close()
