"""GPU parity: QPSKModulator (K3), QPSKDeModulator chain + framer (K5), synthetic channel (K7), BER (K6)
through the C ABI vs the CPU oracle.

Tolerances (north_star): filter / loop outputs max |err| <= 1e-5 * max|y|; demodulated bits, frames
and payloads bit-exact.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REL_TOL = 1e-5

TSC = "11001010011101100100100110101100" + "01110100111001011010001101101001"   # testAtDataLevel.cs:20-22
def test_modulate_frames_dev_more_than_one_grid_of_frames(gpu, orc):
    """Frame batches beyond gridDim.y (65535) go through in slices: 70000 short frames, spot-checked around the seam."""
    import torch
    frames, n_payload = 70000, 6
    m = gpu.QPSKModulator(4000, 1000, 0.35, 6, True, TSC)
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    pay = torch.empty((frames, n_payload), dtype=torch.uint8, device="cuda")
    gpu.fill_bytes_dev(9, 0, frames, n_payload, pay.data_ptr(), s)
    ff = m.frame_floats(n_payload, b"S", b"E")
    out = torch.zeros((frames, ff), dtype=torch.float32, device="cuda")
    assert m.modulate_frames_dev(pay.data_ptr(), n_payload, frames, b"S", b"E", out.data_ptr(), ff, s) == ff
    torch.cuda.synchronize()
    om = orc.QPSKModulator(4000, 1000, 0.35, 6, True, TSC)
    for f in (0, 65534, 65535, 65536, frames - 1):
        want = om.ModulateBytes(pay[f].cpu().numpy().tobytes(), b"S", b"E")
        assert _close(out[f].cpu().numpy(), want), f


def test_full_size_modulator_share_config5(gpu, orc):
    """BASELINE configs[4], one GPU's share at full size (2048 frames x 64 KiB payload, sps 4, span 10: 17.2 GB of
    samples): frames spread over the batch against the oracle, the differential chain restarting per frame (two frames
    given the same payload come out identical wherever they sit), nothing written in the row padding."""
    import torch
    frames, n_payload = 2048, 65536
    fs, rs = 4000, 1000
    m = gpu.QPSKModulator(fs, rs, 0.35, 10, True, TSC)
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    pay = torch.empty((frames, n_payload), dtype=torch.uint8, device="cuda")
    gpu.fill_bytes_dev(7, 0, frames, n_payload, pay.data_ptr(), s)
    torch.cuda.synchronize()
    pay[1500] = pay[3]                                                      # twin frames far apart
    ff = m.frame_floats(n_payload, b"START", b"END")
    stride = ff + 2
    out = torch.empty((frames, stride), dtype=torch.float32, device="cuda")
    out[:, ff:] = 0
    assert m.modulate_frames_dev(pay.data_ptr(), n_payload, frames, b"START", b"END", out.data_ptr(), stride, s) == ff
    torch.cuda.synchronize()
    assert torch.equal(out[1500], out[3])
    assert not out[:, ff:].any()
    om = orc.QPSKModulator(fs, rs, 0.35, 10, True, TSC)
    for f in (0, 1023, frames - 1):
        want = om.ModulateBytes(pay[f].cpu().numpy().tobytes(), b"START", b"END")
        assert want.size == ff
        assert _close(out[f, :ff].cpu().numpy(), want)
    del out


TEXT = "The Quick Brown fox jump yes yes man good!"                                # testAtDataLevel.cs:35
START, STOP = "MESSAGE_START", "MESSAGE_STOP"
ALPHA04 = float(np.float32(0.4))                                                     # const float RRCAlpha = .4f


def _close(got, want, tol=REL_TOL):
    assert got.shape == want.shape, (got.shape, want.shape)
    if want.size == 0:
        return True
    return np.abs(got - want).max() <= tol * max(np.abs(want).max(), 1e-30)


def _bits(n, seed):
    return "".join(np.random.default_rng(seed).choice(["0", "1"], n))


# ---------------------------------------------------------------------------------------------
# modulator
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fs,rs,alpha,span,diff,tsc", [
    (10_000_000, 5_000_000, ALPHA04, 10, True, TSC),       # config 1 (sps 2, 21 taps)
    (4000, 1000, 0.35, 10, True, None),                    # sps 4
    (10_000_000, 10_000_000 // 30, 0.9, 10, True, None),   # testFullDemodChain.cs:18,41 (sps 30, 301 taps)
    (4000, 1000, 0.35, 16, False, "0110"),                 # absolute mapping
    (3000, 1000, 0.5, 5, True, "101"),                     # odd TSC, even-length filter (16 taps)
    (2500, 1000, 0.35, 6, True, None),                     # fs/rs = 2.5: banker's rounding -> 13 taps, sps int-div 2
    (8000, 1000, 0.25, 64, True, None),                    # long filter (513 taps), beta on the singular branch
])
@pytest.mark.parametrize("nbits", [2, 3, 600, 4096, 20001])
def test_modulate_matches_oracle(gpu, orc, fs, rs, alpha, span, diff, tsc, nbits):
    bits = _bits(nbits, nbits + span)
    want_m = orc.QPSKModulator(fs, rs, alpha, span, diff, tsc)
    got_m = gpu.QPSKModulator(fs, rs, alpha, span, diff, tsc)
    assert np.array_equal(want_m.getCoeef(), got_m.getCoeef())
    want = want_m.Modulate(bits)
    got = got_m.Modulate(bits)
    assert _close(got, want)
    # no pulse shaping: the zero-stuffed symbol train is exact (+-1/sqrt2 on the symbol grid)
    want0 = want_m.Modulate(bits, False)
    got0 = got_m.Modulate(bits, False)
    assert np.array_equal(got0.view(np.uint32), want0.view(np.uint32))


def test_modulate_edge_cases(gpu, orc):
    for mod in (gpu, orc):
        m = mod.QPSKModulator(4000, 1000, 0.35, 6)
        assert m.Modulate("").size == 0
        assert m.Modulate("1").size == 0                                  # odd trailing bit dropped (:112-113)
        with pytest.raises(mod.ArgumentNullException):
            m.Modulate(None)
        with pytest.raises(mod.ArgumentException):
            m.ModulateBytes(b"abc", b"", b"E")                            # :60
        with pytest.raises(mod.ArgumentException):
            m.ModulateBytes(b"abc", b"S", b"")                            # :61
    # characters other than '0'/'1' follow the reference's `c - '0'` arithmetic
    weird = "01x10 1z00y1"
    for diff in (True, False):
        a = orc.QPSKModulator(4000, 1000, 0.35, 6, diff).Modulate(weird)
        b = gpu.QPSKModulator(4000, 1000, 0.35, 6, diff).Modulate(weird)
        assert _close(b, a)
    # whitespace TSC counts as no TSC (:27)
    a = orc.QPSKModulator(4000, 1000, 0.35, 6, True, "  ").Modulate("0110")
    b = gpu.QPSKModulator(4000, 1000, 0.35, 6, True, "  ").Modulate("0110")
    assert _close(b, a)


def test_modulate_bytes_and_text(gpu, orc):
    want = orc.QPSKModulator(10_000_000, 5_000_000, ALPHA04, 10, tsc=TSC).ModulateTextUtf8(TEXT, START, STOP)
    got = gpu.QPSKModulator(10_000_000, 5_000_000, ALPHA04, 10, tsc=TSC).ModulateTextUtf8(TEXT, START, STOP)
    assert want.size == 2 * 620                                            # SURVEY §4: 620 complex samples per burst
    assert _close(got, want)
    rng = np.random.default_rng(3)
    payload = rng.integers(0, 256, 5000, dtype=np.uint8).tobytes()
    for tsc in (None, "101", TSC):
        a = orc.QPSKModulator(4000, 1000, 0.35, 10, True, tsc).ModulateBytes(payload, b"\x02", b"\x03")
        b = gpu.QPSKModulator(4000, 1000, 0.35, 10, True, tsc).ModulateBytes(payload, b"\x02", b"\x03")
        assert _close(b, a)


def test_modulate_frames_dev_batch(gpu, orc):
    """config 5 shape at test size: [frames][payload] device bytes -> [frames][samples]."""
    import torch
    frames, n_payload = 9, 3000
    m = gpu.QPSKModulator(4000, 1000, 0.35, 10, True, TSC)
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    pay = torch.empty((frames, n_payload), dtype=torch.uint8, device="cuda")
    gpu.fill_bytes_dev(5, 100, frames, n_payload, pay.data_ptr(), s)
    ff = m.frame_floats(n_payload, b"START", b"END")
    stride = ff + 6
    out = torch.zeros((frames, stride), dtype=torch.float32, device="cuda")
    assert m.modulate_frames_dev(pay.data_ptr(), n_payload, frames, b"START", b"END", out.data_ptr(), stride, s) == ff
    torch.cuda.synchronize()
    pay_h = pay.cpu().numpy()
    out_h = out.cpu().numpy()
    om = orc.QPSKModulator(4000, 1000, 0.35, 10, True, TSC)
    for f in range(frames):
        # payload generator: byte k of channel c = top byte of rng(seed, 4c+3, k)
        want_pay = np.array([orc.rng_u64(5, 4 * (100 + f) + 3, k) >> 56 for k in range(0, n_payload, 499)], np.uint8)
        assert np.array_equal(pay_h[f, ::499], want_pay)
        want = om.ModulateBytes(pay_h[f].tobytes(), b"START", b"END")
        assert want.size == ff
        assert _close(out_h[f, :ff], want)
        assert not out_h[f, ff:].any()                                      # nothing written past the frame


@pytest.mark.parametrize("n_payload,start", [(3001, b"S"), (3002, b"ST"), (3003, b"STA"), (2999, b"STAR"), (4097, b"STARTS")])
def test_modulate_frames_dev_alignments(gpu, orc, n_payload, start):
    """The differential pre-pass sums interior tiles as 32-bit words: every byte alignment of the tile start
    (row pitch and start-marker length both shift it) must give the oracle's symbols."""
    import torch
    frames = 5
    m = gpu.QPSKModulator(4000, 1000, 0.35, 10, True, TSC)
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    pay = torch.empty((frames, n_payload), dtype=torch.uint8, device="cuda")
    gpu.fill_bytes_dev(6, 7, frames, n_payload, pay.data_ptr(), s)
    ff = m.frame_floats(n_payload, start, b"END")
    out = torch.zeros((frames, ff), dtype=torch.float32, device="cuda")
    assert m.modulate_frames_dev(pay.data_ptr(), n_payload, frames, start, b"END", out.data_ptr(), ff, s) == ff
    torch.cuda.synchronize()
    pay_h, out_h = pay.cpu().numpy(), out.cpu().numpy()
    om = orc.QPSKModulator(4000, 1000, 0.35, 10, True, TSC)
    for f in range(frames):
        assert _close(out_h[f], om.ModulateBytes(pay_h[f].tobytes(), start, b"END"))


def test_modulator_linearity_of_frames(gpu):
    """Full-size property (no oracle): every frame of a large batch equals the same frame done alone."""
    import torch
    frames, n_payload = 64, 65536
    m = gpu.QPSKModulator(4000, 1000, 0.35, 10, True, TSC)
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    pay = torch.empty((frames, n_payload), dtype=torch.uint8, device="cuda")
    gpu.fill_bytes_dev(9, 0, frames, n_payload, pay.data_ptr(), s)
    ff = m.frame_floats(n_payload, b"S", b"E")
    out = torch.empty((frames, ff), dtype=torch.float32, device="cuda")
    m.modulate_frames_dev(pay.data_ptr(), n_payload, frames, b"S", b"E", out.data_ptr(), ff, s)
    one = torch.empty((1, ff), dtype=torch.float32, device="cuda")
    for f in (0, 17, 63):
        m.modulate_frames_dev(pay[f].data_ptr(), n_payload, 1, b"S", b"E", one.data_ptr(), ff, s)
        torch.cuda.synchronize()
        assert torch.equal(one[0], out[f])
    # pulse peaks: sampling the output on the symbol grid with a matched filter is tested in the chain tests


# ---------------------------------------------------------------------------------------------
# demodulator: config 1 (testAtDataLevel) — K consecutive bursts through one persistent demod
# ---------------------------------------------------------------------------------------------
def _datalevel_bursts(orc, k, seed=7):
    fs = 10_000_000
    mod = orc.QPSKModulator(fs, fs // 2, ALPHA04, 10, tsc=TSC)
    tx = orc.NCO(100e6, fs, 1, seed=seed, stream=0)
    rx = orc.NCO(100e6, fs, 1, seed=seed, stream=1)
    out = []
    for _ in range(k):
        s = mod.ModulateTextUtf8(TEXT, START, STOP)
        out.append(orc.channel_apply(tx, rx, 0, s))
    return out


@pytest.mark.parametrize("fir_mode", ["exact", "fast"])
def test_datalevel_roundtrip_matches_oracle(gpu, orc, fir_mode):
    fs = 10_000_000
    bursts = _datalevel_bursts(orc, 8)
    od = orc.QPSKDeModulator(fs, fs // 2, ALPHA04, 10, tsc=TSC)
    gd = gpu.QPSKDeModulator(fs, fs // 2, ALPHA04, 10, tsc=TSC)
    gd.set_fir_mode(gpu.FIR_EXACT if fir_mode == "exact" else gpu.FIR_FAST)
    texts = []
    for y in bursts:
        want = od.DeModulateTextUtf8(y, START, STOP)
        got = gd.DeModulateTextUtf8(y, START, STOP)
        assert got == want
        texts.append(got)
        assert gd.in_frame == od.in_frame
    assert texts[0] == "" and all(t == TEXT for t in texts[1:])          # SURVEY §4 open question (a): first burst is lost
    ws, gs = od.loop_state(), gd.loop_state()
    for k in ("costas_theta", "costas_freq", "mm_mu", "mm_integral"):
        assert abs(ws[k] - gs[k]) <= 1e-5 * max(1.0, abs(ws[k])), k


@pytest.mark.parametrize("fir_mode", ["exact", "fast"])
def test_datalevel_bits_and_constellation(gpu, orc, fir_mode):
    fs = 10_000_000
    bursts = _datalevel_bursts(orc, 5, seed=11)
    od, od2 = (orc.QPSKDeModulator(fs, fs // 2, ALPHA04, 10, tsc=TSC) for _ in range(2))
    gd, gd2 = (gpu.QPSKDeModulator(fs, fs // 2, ALPHA04, 10, tsc=TSC) for _ in range(2))
    for g in (gd, gd2):
        g.set_fir_mode(gpu.FIR_EXACT if fir_mode == "exact" else gpu.FIR_FAST)
    for y in bursts:
        assert gd.DeModulate(y) == od.DeModulate(y)                        # bits bit-exact
        wc, gc = od2.deModulateConstellation(y), gd2.deModulateConstellation(y)
        assert _close(gc, wc)
        if fir_mode == "exact":
            assert np.array_equal(gc.view(np.uint32), wc.view(np.uint32))


def test_demod_chunked_stream_equals_one_shot(gpu, orc):
    """All state persists across calls: arbitrary chunking gives the same bits (SURVEY §3.2)."""
    fs, rs = 4000, 1000
    mod = orc.QPSKModulator(fs, rs, 0.35, 10)
    x = np.concatenate([mod.Modulate(_bits(3000, 50 + i)) for i in range(3)])
    od = orc.QPSKDeModulator(fs, rs, 0.35, 10, SymbolSyncBandwith=0.002)
    g1 = gpu.QPSKDeModulator(fs, rs, 0.35, 10, SymbolSyncBandwith=0.002)
    g2 = gpu.QPSKDeModulator(fs, rs, 0.35, 10, SymbolSyncBandwith=0.002)
    for g in (g1, g2):
        g.set_fir_mode(gpu.FIR_EXACT)
    want = od.DeModulate(x)
    one = g1.DeModulate(x)
    cuts = [0, 2, 10, 1000, 1002, 7778, 20000, x.size]
    many = "".join(g2.DeModulate(x[a:b]) for a, b in zip(cuts[:-1], cuts[1:]))
    assert one == want
    assert many == want


@pytest.mark.parametrize("diff", [True, False])
@pytest.mark.parametrize("sps,span", [(4, 10), (2, 10), (8, 6)])
def test_demod_bits_no_tsc(gpu, orc, diff, sps, span):
    fs, rs = sps * 1000, 1000
    bits = _bits(4096, sps + span)
    x = orc.QPSKModulator(fs, rs, 0.35, span, diff).Modulate(bits)
    z = (x[0::2] + 1j * x[1::2]) * np.exp(1j * (0.4 + 2e-4 * np.arange(x.size // 2)))
    rng = np.random.default_rng(1)
    z = z + 0.02 * (rng.standard_normal(z.size) + 1j * rng.standard_normal(z.size))
    y = np.empty_like(x)
    y[0::2], y[1::2] = z.real, z.imag
    od = orc.QPSKDeModulator(fs, rs, 0.35, span, 0.002, 120.0, differentialEncoding=diff)
    gd = gpu.QPSKDeModulator(fs, rs, 0.35, span, 0.002, 120.0, differentialEncoding=diff)
    gd.set_fir_mode(gpu.FIR_EXACT)
    want, got = od.DeModulate(y), gd.DeModulate(y)
    assert got == want
    assert len(got) > 3000


def test_demod_full_chain_with_fll_matches_oracle(gpu, orc):
    """config 3 at test size: FLL -> MF -> MM -> Costas -> decode, parameters of testFullDemodChain.cs."""
    fs = 10_000_000
    rs = fs // 30
    bits = _bits(1024, 77)
    x = orc.QPSKModulator(fs, rs, 0.9, 10).Modulate(bits)
    tx = orc.NCO(935e6, fs, 20, 120, seed=3, stream=0)
    rx = orc.NCO(935e6, fs, 10, 30, seed=3, stream=1)
    noise = orc.noise_iq(-40.0, x.size // 2, 3, 2)
    y = orc.channel_apply(tx, rx, 1, x, noise)
    kw = dict(RrcAlpha=float(np.float32(0.9)), rrcSpan=11, SymbolSyncBandwith=0.001, CostasLoopBandwith=10.0,
              CFOLoopBandwith=float(np.float32(0.01)), use_fll=True)
    od = orc.QPSKDeModulator(fs, rs, **kw)
    gd = gpu.QPSKDeModulator(fs, rs, **kw)
    gd.set_fir_mode(gpu.FIR_EXACT)
    half = (y.size // 4) * 2
    want = od.DeModulate(y[:half]) + od.DeModulate(y[half:])
    got = gd.DeModulate(y[:half]) + gd.DeModulate(y[half:])
    assert got == want
    ws, gs = od.loop_state(), gd.loop_state()
    assert abs(ws["fll_freq"] - gs["fll_freq"]) <= 1e-5 * max(abs(ws["fll_freq"]), 1e-3)
    assert abs(ws["costas_theta"] - gs["costas_theta"]) <= 1e-5 * max(1.0, abs(ws["costas_theta"]))


def test_demod_fll_time_chunk_pipeline_matches_oracle(gpu, orc):
    """256 channels x 5700 samples with the FLL on: bits_dev splits the call into time chunks (FLL -> MF of chunk t+1 on
    a side stream, MM -> Costas -> decode of chunk t on the caller's).  Every channel must still equal its own
    single-stream oracle, over two calls (state carried), with a call length that is not a multiple of the chunk."""
    fs, rs, Cn = 2000, 1000, 256
    rng = np.random.default_rng(11)
    rows = []
    for c in range(Cn):
        payload = bytes(rng.integers(0, 256, 700, dtype=np.uint8))
        x = orc.QPSKModulator(fs, rs, 0.35, 10, True, TSC).ModulateBytes(payload, b"<<", b">>")
        z = (x[0::2] + 1j * x[1::2]) * np.exp(1j * (0.05 * c + 2e-4 * (c % 17) * np.arange(x.size // 2)))
        z = z + 0.01 * (rng.standard_normal(z.size) + 1j * rng.standard_normal(z.size))
        y = np.empty_like(x)
        y[0::2], y[1::2] = z.real, z.imag
        rows.append(y)
    L = min(r.size for r in rows)
    Y = np.stack([r[:L] for r in rows]).astype(np.float32)
    assert L // 2 >= 5000
    kw = dict(RrcAlpha=float(np.float32(0.35)), rrcSpan=10, SymbolSyncBandwith=0.002, CostasLoopBandwith=120.0,
              CFOLoopBandwith=float(np.float32(0.01)), use_fll=True)   # no TSC strip: the raw bit stream is compared
    gd = gpu.QPSKDeModulator(fs, rs, channels=Cn, **kw)
    gd.set_fir_mode(gpu.FIR_EXACT)
    cut = 2 * 2237                                    # both calls are long enough to be split (>= 2048 samples)
    got = [gd.DeModulate(np.ascontiguousarray(Y[:, :cut])), gd.DeModulate(np.ascontiguousarray(Y[:, cut:]))]
    bad = 0
    for c in range(Cn):
        od = orc.QPSKDeModulator(fs, rs, **kw)
        want = [od.DeModulate(Y[c, :cut]), od.DeModulate(Y[c, cut:])]
        bad += (want[0] != got[0][c]) + (want[1] != got[1][c])
    assert bad == 0
    assert min(len(g) for g in got[0]) > 2000 and min(len(g) for g in got[1]) > 2000


def test_demod_batch_channels_match_single_streams(gpu, orc):
    fs, rs, Cn = 4000, 1000, 6
    xs = []
    for c in range(Cn):
        x = orc.QPSKModulator(fs, rs, 0.35, 10, True, TSC).ModulateBytes(bytes(range(40 + c, 140 + c)), b"<<", b">>")
        z = (x[0::2] + 1j * x[1::2]) * np.exp(1j * (0.1 * c + 1e-4 * c * np.arange(x.size // 2)))
        y = np.empty_like(x)
        y[0::2], y[1::2] = z.real, z.imag
        xs.append(y)
    X = np.stack(xs)
    kw = dict(RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002, tsc=TSC)
    gd = gpu.QPSKDeModulator(fs, rs, channels=Cn, max_frame_bytes=4096, **kw)
    gd.set_fir_mode(gpu.FIR_EXACT)
    ods = [orc.QPSKDeModulator(fs, rs, **kw) for _ in range(Cn)]
    for rep in range(3):                                                   # state carried burst to burst
        got = gd.DeModulateBytes(X, b"<<", b">>")
        for c in range(Cn):
            assert got[c] == ods[c].DeModulateBytes(X[c], b"<<", b">>"), (rep, c)
    assert any(len(g) for g in got)


# ---------------------------------------------------------------------------------------------
# framer
# ---------------------------------------------------------------------------------------------
def _clean_stream(orc, payloads, sm, em, fs=4000, rs=1000, tsc=None, gap_bits=64):
    mod = orc.QPSKModulator(fs, rs, 0.35, 10, True, tsc)
    return np.concatenate([mod.ModulateBytes(p, sm, em) for p in payloads])


def test_framer_marker_spanning_calls_and_offsets(gpu, orc):
    """Item 11 of the SURVEY §4 checklist: offset hunt, carry of 8*len+7 bits, payload before the end marker."""
    fs, rs = 4000, 1000
    sm, em = b"\xa5START\x5a", b"\x5aSTOP\xa5"
    rng = np.random.default_rng(8)
    payloads = [rng.integers(0, 256, n, dtype=np.uint8).tobytes() for n in (10, 300, 1, 57)]
    x = _clean_stream(orc, payloads, sm, em)
    kw = dict(RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002)
    for chunk in (x.size, 2 * 997, 2 * 150, 2 * 41):
        od = orc.QPSKDeModulator(fs, rs, **kw)
        gd = gpu.QPSKDeModulator(fs, rs, max_frame_bytes=1024, **kw)
        gd.set_fir_mode(gpu.FIR_EXACT)
        got_all, want_all = [], []
        for a in range(0, x.size, chunk):
            w = od.DeModulateBytes(x[a:a + chunk], sm, em)
            g = gd.DeModulateBytes(x[a:a + chunk], sm, em)
            assert g == w, (chunk, a)
            assert gd.in_frame == od.in_frame
            if w:
                want_all.append(w)
                got_all.append(g)
        assert got_all == want_all
        if chunk >= 2 * 997:
            assert any(w in payloads for w in want_all)


def test_framer_ring_overflow_resets(gpu, orc):
    fs, rs = 4000, 1000
    sm, em = b"AB", b"YZ"
    x = _clean_stream(orc, [bytes(200), b"ok-after-overflow"], sm, em)
    kw = dict(RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002)
    od = orc.QPSKDeModulator(fs, rs, ring_capacity=64, **kw)
    gd = gpu.QPSKDeModulator(fs, rs, max_frame_bytes=64, **kw)
    gd.set_fir_mode(gpu.FIR_EXACT)
    for a in range(0, x.size, 2 * 500):
        assert gd.DeModulateBytes(x[a:a + 1000], sm, em) == od.DeModulateBytes(x[a:a + 1000], sm, em)
        assert gd.in_frame == od.in_frame


def _framer_streams(rng, channels, sm, em, max_payload=40):
    bits_of = lambda b: "".join(format(v, "08b") for v in b)
    rows = []
    for _ in range(channels):
        t = ""
        for _f in range(int(rng.integers(1, 6))):
            t += "".join(rng.choice(["0", "1"], int(rng.integers(0, 50))))
            body = rng.integers(0, 256, int(rng.integers(0, max_payload)), dtype=np.uint8).tobytes()
            if rng.random() < 0.3:
                body = body[: len(body) // 2] + sm + body[len(body) // 2:]      # a start marker inside the payload
            t += bits_of(sm + body + em)
        t += "".join(rng.choice(["0", "1"], int(rng.integers(0, 50))))
        rows.append(t)
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("channels,markers,ring", [(1, (b"S", b"E"), 1 << 20), (5, (b"\xa5START\x5a", b"\x5aSTOP\xa5"), 1 << 20),
                                                   (37, (b"AB", b"YZ"), 24), (130, (b"\x00", b"\xff\xff"), 1 << 20),
                                                   (3, (bytes(range(1, 41)), b"\x7e"), 16)])
def test_framer_on_bits_ragged_channels(gpu, orc, channels, markers, ring):
    """The warp-per-channel framer kernel on its own (QPSKDeModulator.cs:179-259): ragged per-channel bit chunks
    (including empty ones), frames at every bit offset, markers split across calls, start markers inside payloads, ring
    overflow -> reset; payloads and the in-frame flag must equal the oracle's after every call."""
    sm, em = markers
    rng = np.random.default_rng(100 + channels)
    rows = _framer_streams(rng, channels, sm, em)
    gd = gpu.QPSKDeModulator(4000, 1000, max_frame_bytes=ring, channels=channels)
    ods = [orc.QPSKDeModulator(4000, 1000, ring_capacity=ring) for _ in range(channels)]
    pos = [0] * channels
    got_frames = 0
    while any(pos[c] < len(rows[c]) for c in range(channels)):
        big = rng.random() < 0.2
        take = [int(rng.integers(0, 400 if big else 70)) for _ in range(channels)]
        chunks = [rows[c][pos[c]:pos[c] + take[c]] for c in range(channels)]
        pos = [pos[c] + take[c] for c in range(channels)]
        got = gd.FrameBits(chunks if channels > 1 else chunks[0], sm, em, cap=4096)
        got = got if channels > 1 else [got]
        for c in range(channels):
            want = ods[c].FrameBits(chunks[c], sm, em, cap=4096)
            assert got[c] == want, (c, pos[c])
            got_frames += bool(want)
        inf = np.atleast_1d(gd.in_frame)
        assert [bool(v) for v in inf] == [bool(o.in_frame) for o in ods]
    assert got_frames > 0 or ring < 64


@pytest.mark.gpu
def test_framer_on_bits_long_call(gpu, orc):
    """One call holding many frames' worth of bits (only the first frame comes out, the rest is dropped exactly as the
    reference drops it, :226-229) and a frame that spans three calls."""
    sm, em = b"<<", b">>"
    rng = np.random.default_rng(5)
    bits_of = lambda b: "".join(format(v, "08b") for v in b)
    payloads = [rng.integers(0, 256, n, dtype=np.uint8).tobytes() for n in (700, 3, 1500)]
    t = "101" + "".join(bits_of(sm + p + em) + "0110" for p in payloads)
    gd, od = gpu.QPSKDeModulator(4000, 1000), orc.QPSKDeModulator(4000, 1000)
    assert gd.FrameBits(t, sm, em, cap=8192) == od.FrameBits(t, sm, em, cap=8192) == payloads[0]
    long_frame = "1" * 5 + bits_of(sm + bytes(range(256)) * 20 + em)
    third = len(long_frame) // 3
    for a in (0, third, 2 * third):
        part = long_frame[a:a + third] if a < 2 * third else long_frame[a:]
        g, w = gd.FrameBits(part, sm, em, cap=8192), od.FrameBits(part, sm, em, cap=8192)
        assert g == w
        assert gd.in_frame == od.in_frame
    assert w == bytes(range(256)) * 20


@pytest.mark.gpu
def test_text_default_markers_roundtrip(gpu, orc):
    """Default STX / ETX markers (QPSKModulator.cs:76-77, QPSKDeModulator.cs:264-265) through both text calls."""
    fs, rs = 4000, 1000
    gm, om = gpu.QPSKModulator(fs, rs, 0.35, 10), orc.QPSKModulator(fs, rs, 0.35, 10)
    x = om.ModulateTextUtf8("warm-up burst")
    y = om.ModulateTextUtf8("héllo, wörld")
    assert _close(gm.ModulateTextUtf8("héllo, wörld"), y)
    assert _close(gm.ModulateTextUtf8("héllo, wörld", "\x02", "\x03"), y)
    kw = dict(RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002)
    gd, od = gpu.QPSKDeModulator(fs, rs, **kw), orc.QPSKDeModulator(fs, rs, **kw)
    gd.set_fir_mode(gpu.FIR_EXACT)
    for burst in (x, y, y):
        assert gd.DeModulateTextUtf8(burst) == od.DeModulateTextUtf8(burst)


def test_demod_error_behaviour(gpu, orc):
    for mod in (gpu, orc):
        d = mod.QPSKDeModulator(4000, 1000)
        with pytest.raises(mod.ArgumentException):
            d.DeModulate(np.zeros(3, np.float32))                          # odd length (:347-348)
        with pytest.raises(mod.ArgumentException):
            d.DeModulateBytes(np.zeros(4, np.float32), b"", b"x")          # :174
        with pytest.raises(mod.ArgumentException):
            d.DeModulateBytes(np.zeros(4, np.float32), b"x", b"")          # :175
        assert d.DeModulate(np.zeros(0, np.float32)) == ""                 # :350-351
        assert d.DeModulateBytes(np.zeros(0, np.float32), b"a", b"b") == b""
    with pytest.raises(gpu.ArgumentOutOfRangeException):
        gpu.QPSKDeModulator(4000, 1000, CFOLoopBandwith=0.0)               # FLL ctor check (Band-Edge Filter.cs:45)
    with pytest.raises(orc.ArgumentOutOfRangeException):
        orc.QPSKDeModulator(4000, 1000, CFOLoopBandwith=0.0)


# ---------------------------------------------------------------------------------------------
# channel simulator, BER
# ---------------------------------------------------------------------------------------------
def _ulp_diff(a, b):
    ai = a.view(np.int32).astype(np.int64)
    bi = b.view(np.int32).astype(np.int64)
    ai = np.where(ai < 0, -(ai & 0x7FFFFFFF), ai)
    bi = np.where(bi < 0, -(bi & 0x7FFFFFFF), bi)
    return np.abs(ai - bi)


@pytest.mark.parametrize("mode,noise", [(0, -1000.0), (1, -1000.0), (1, -30.0)])
def test_channel_matches_oracle(gpu, orc, mode, noise):
    fs = 10_000_000
    x = orc.fill_uniform(2, 9, 0, 2 * 30000)
    Cn, first, seed = 3, 5, 1234
    ch = gpu.SimChannel(935e6, 935e6, fs, 20, 10, 120.0, 30.0, noise_dbfs=noise, mode=mode, seed=seed, channels=Cn,
                        first_channel=first)
    X = np.stack([x] * Cn)
    got = np.concatenate([ch.apply(X[:, :2 * 12345]), ch.apply(X[:, 2 * 12345:])], axis=1)   # state persists
    for c in range(Cn):
        k = first + c
        tx = orc.NCO(935e6, fs, 20, 120.0, seed=seed, stream=4 * k)
        rx = orc.NCO(935e6, fs, 10, 30.0, seed=seed, stream=4 * k + 1)
        nz = orc.noise_iq(noise, x.size // 2, seed, 4 * k + 2) if noise > -300 else None
        want = orc.channel_apply(tx, rx, mode, x, nz)
        # CUDA's fp64 sin/cos/log are within 1-2 ulp of glibc's: after the cast to fp32 nearly every
        # sample is identical and none differs by more than one fp32 ulp
        d = _ulp_diff(got[c], want)
        assert d.max() <= 1, d.max()
        assert (d != 0).mean() < 1e-3
    assert not np.array_equal(got[0], got[1])                              # channels have their own LO errors


def test_channel_multipath_matches_oracle(gpu, orc):
    fs = 1_000_000
    x = orc.fill_uniform(3, 1, 0, 2 * 5000)
    gains = [1.0, 0.0, 0.3, -0.2, -0.1, 0.25]
    delays = [0, 3, 17]
    ch = gpu.SimChannel(0.0, 0.0, fs, 0, 0, mode=0, path_gains_iq=gains, path_delays=delays, seed=1)
    got = np.concatenate([ch.apply(x[:2 * 10]), ch.apply(x[2 * 10:2 * 2000]), ch.apply(x[2 * 2000:])])
    mp = orc.multipath(x, gains, delays)
    tx = orc.NCO(0.0, fs, 0, 0.0, seed=1, stream=0)
    rx = orc.NCO(0.0, fs, 0, 0.0, seed=1, stream=1)
    want = orc.channel_apply(tx, rx, 0, mp)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))      # zero-ppm NCOs: phase stays 0, exact


def test_ber_counters_and_unpack(gpu):
    import torch
    rng = np.random.default_rng(4)
    Cn, nref = 5, 1000
    ref_bytes = rng.integers(0, 256, (Cn, nref // 8), dtype=np.uint8)
    ref_bits = np.unpackbits(ref_bytes, axis=1)
    rx = ref_bits.copy()
    n_rx = np.array([1000, 1000, 900, 1100, 0], np.int64)
    rx = np.concatenate([rx, rng.integers(0, 2, (Cn, 200), dtype=np.uint8)], axis=1)
    flips = [0, 13, 7, 2, 0]
    for c, k in enumerate(flips):
        idx = rng.choice(min(n_rx[c], nref) or 1, k, replace=False)
        rx[c, idx] ^= 1
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    d_bytes = torch.from_numpy(ref_bytes).cuda()
    d_ref = torch.empty((Cn, nref), dtype=torch.uint8, device="cuda")
    gpu.unpack_bits_dev(d_bytes.data_ptr(), nref // 8, nref // 8, Cn, d_ref.data_ptr(), nref, s)
    torch.cuda.synchronize()
    assert np.array_equal(d_ref.cpu().numpy(), ref_bits)
    d_rx = torch.from_numpy(rx).cuda()
    d_n = torch.from_numpy(n_rx).cuda()
    cnt = torch.zeros((Cn, 2), dtype=torch.int32, device="cuda")
    gpu.ber_count_dev(d_rx.data_ptr(), rx.shape[1], d_n.data_ptr(), d_ref.data_ptr(), nref, nref, Cn, cnt.data_ptr(), s)
    torch.cuda.synchronize()
    got = cnt.cpu().numpy()
    want_err = [0, 13, 7 + 100, 2, 1000]
    assert got[:, 0].tolist() == want_err
    assert got[:, 1].tolist() == [nref] * Cn


@pytest.mark.parametrize("rx_stride,ref_stride,n_ref", [(1203, 1001, 997), (1202, 1000, 1000), (1201, 1003, 999), (1207, 1006, 3)])
def test_ber_counters_unaligned_rows(gpu, rx_stride, ref_stride, n_ref):
    """ber_kernel compares word-wise with funnel shifts: odd row pitches put every channel's rx / ref row at a
    different byte alignment; arbitrary byte values (not only 0/1) must still compare as bytes."""
    import torch
    rng = np.random.default_rng(rx_stride)
    Cn = 9
    ref = rng.integers(0, 256, (Cn, ref_stride), dtype=np.uint8)
    rx = rng.integers(0, 256, (Cn, rx_stride), dtype=np.uint8)
    n_rx = rng.integers(0, n_ref + 40, Cn).astype(np.int64)
    n_rx[0], n_rx[1] = n_ref, 0
    for c in range(Cn):
        m = int(min(n_rx[c], n_ref))
        rx[c, :m] = ref[c, :m]
        if m:
            idx = rng.choice(m, min(m, 5 + c), replace=False)
            rx[c, idx] ^= rng.integers(1, 256, idx.size, dtype=np.uint8)
    want = [int((rx[c, :min(n_rx[c], n_ref)] != ref[c, :min(n_rx[c], n_ref)]).sum() + max(0, n_ref - n_rx[c])) for c in range(Cn)]
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    d_rx, d_ref, d_n = torch.from_numpy(rx).cuda(), torch.from_numpy(ref).cuda(), torch.from_numpy(n_rx).cuda()
    cnt = torch.zeros((Cn, 2), dtype=torch.int32, device="cuda")
    gpu.ber_count_dev(d_rx.data_ptr(), rx_stride, d_n.data_ptr(), d_ref.data_ptr(), ref_stride, n_ref, Cn, cnt.data_ptr(), s)
    torch.cuda.synchronize()
    got = cnt.cpu().numpy()
    assert got[:, 0].tolist() == want
    assert got[:, 1].tolist() == [n_ref] * Cn


def test_batched_chain_device_resident_ber(gpu, orc):
    """config 3/4 at test size, fully device-resident: payload -> modulate -> channel -> demod -> BER.
    Parameters of testAtDataLevel.cs (the configuration in which the reference loops lock)."""
    import torch
    fs = 10_000_000
    rs = fs // 2
    Cn, n_payload, seed = 40, 64, 21
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    mod = gpu.QPSKModulator(fs, rs, ALPHA04, 10, True, TSC)
    pay = torch.empty((Cn, n_payload), dtype=torch.uint8, device="cuda")
    gpu.fill_bytes_dev(seed, 0, Cn, n_payload, pay.data_ptr(), s)
    ff = mod.frame_floats(n_payload, b"S", b"E")
    tx = torch.empty((Cn, ff), dtype=torch.float32, device="cuda")
    mod.modulate_frames_dev(pay.data_ptr(), n_payload, Cn, b"S", b"E", tx.data_ptr(), ff, s)
    ch = gpu.SimChannel(100e6, 100e6, fs, 1, 1, noise_dbfs=-40.0, mode=1, seed=seed, channels=Cn)
    rxs = torch.empty_like(tx)
    kw = dict(RrcAlpha=ALPHA04, rrcSpan=10, tsc=TSC)
    dem = gpu.QPSKDeModulator(fs, rs, channels=Cn, **kw)
    dem.set_fir_mode(gpu.FIR_EXACT)
    cap = dem.bits_bound(ff)
    bits = torch.zeros((Cn, cap), dtype=torch.uint8, device="cuda")
    nb = torch.zeros(Cn, dtype=torch.int64, device="cuda")
    nref = 8 * (n_payload + 2)
    ref = torch.empty((Cn, nref), dtype=torch.uint8, device="cuda")
    framed = torch.cat([torch.full((Cn, 1), ord("S"), dtype=torch.uint8, device="cuda"), pay,
                        torch.full((Cn, 1), ord("E"), dtype=torch.uint8, device="cuda")], dim=1).contiguous()
    gpu.unpack_bits_dev(framed.data_ptr(), n_payload + 2, n_payload + 2, Cn, ref.data_ptr(), nref, s)
    cnt = torch.zeros((Cn, 2), dtype=torch.int32, device="cuda")
    check = (0, 7, Cn - 1)
    ods = {c: orc.QPSKDeModulator(fs, rs, **kw) for c in check}
    ref_h = None
    for burst in range(4):                                                 # the first bursts are acquisition
        ch.apply_dev(tx.data_ptr(), ff, ff, rxs.data_ptr(), ff, s)
        dem.demod_bits_dev(rxs.data_ptr(), ff, ff, bits.data_ptr(), cap, nb.data_ptr(), s)
        gpu.ber_count_dev(bits.data_ptr(), cap, nb.data_ptr(), ref.data_ptr(), nref, nref, Cn, cnt.data_ptr(), s)
        torch.cuda.synchronize()
        rx_h, bits_h, nb_h, cnt_h = rxs.cpu().numpy(), bits.cpu().numpy(), nb.cpu().numpy(), cnt.cpu().numpy()
        ref_h = ref.cpu().numpy() if ref_h is None else ref_h
        for c, od in ods.items():                                          # bits identical to the oracle's on the same samples
            want = od.DeModulate(rx_h[c])
            got = "".join("1" if b else "0" for b in bits_h[c, : nb_h[c]])
            assert got == want, (burst, c)
            n = min(len(want), nref)
            err = sum(a != str(b) for a, b in zip(want[:n], ref_h[c, :n])) + (nref - n)
            assert cnt_h[c].tolist() == [err, nref], (burst, c)
    assert (cnt_h[:, 1] == nref).all()
    assert (cnt_h[:, 0] == 0).mean() > 0.9, cnt_h[:, 0]                    # locked channels decode error-free


@pytest.mark.parametrize("use_fll", [False, True])
def test_full_size_channel_set_config4(gpu, orc, use_fll):
    """BASELINE configs[3] at full size on one GPU: 16384 impaired channels (config 3's 1024 bursts are a subset), device
    resident end to end.  No oracle run at this size, so: (i) oracle bits on a few channels spread over the set, every
    burst; (ii) batch-position independence — a block of channels cut out of the set and run through a fresh 48-channel
    demodulator gives the same bits and counts; (iii) the BER counters equal a host recount; (iv) locked channels
    decode error-free."""
    import torch
    fs = 10_000_000
    rs = fs // 2
    Cn, n_payload, seed = 16384, 512, 33
    lo, hi = 9001, 9049                                                    # the cut-out block (straddles CTA boundaries)
    ts = torch.cuda.Stream()
    torch.cuda.set_stream(ts)
    s = ts.cuda_stream
    mod = gpu.QPSKModulator(fs, rs, ALPHA04, 10, True, TSC)
    pay = torch.empty((Cn, n_payload), dtype=torch.uint8, device="cuda")
    gpu.fill_bytes_dev(seed, 0, Cn, n_payload, pay.data_ptr(), s)
    ff = mod.frame_floats(n_payload, b"S", b"E")
    tx = torch.empty((Cn, ff), dtype=torch.float32, device="cuda")
    mod.modulate_frames_dev(pay.data_ptr(), n_payload, Cn, b"S", b"E", tx.data_ptr(), ff, s)
    ch = gpu.SimChannel(100e6, 100e6, fs, 1, 1, noise_dbfs=-40.0, mode=1, seed=seed, channels=Cn)
    rxs = torch.empty_like(tx)
    kw = dict(RrcAlpha=ALPHA04, rrcSpan=10, tsc=TSC, use_fll=use_fll)
    dem = gpu.QPSKDeModulator(fs, rs, channels=Cn, **kw)
    sub = gpu.QPSKDeModulator(fs, rs, channels=hi - lo, **kw)
    dem.set_fir_mode(gpu.FIR_EXACT)
    sub.set_fir_mode(gpu.FIR_EXACT)
    cap = dem.bits_bound(ff)
    bits = torch.zeros((Cn, cap), dtype=torch.uint8, device="cuda")
    nb = torch.zeros(Cn, dtype=torch.int64, device="cuda")
    sbits = torch.zeros((hi - lo, cap), dtype=torch.uint8, device="cuda")
    snb = torch.zeros(hi - lo, dtype=torch.int64, device="cuda")
    nref = 8 * (n_payload + 2)
    ref = torch.empty((Cn, nref), dtype=torch.uint8, device="cuda")
    framed = torch.cat([torch.full((Cn, 1), ord("S"), dtype=torch.uint8, device="cuda"), pay,
                        torch.full((Cn, 1), ord("E"), dtype=torch.uint8, device="cuda")], dim=1).contiguous()
    gpu.unpack_bits_dev(framed.data_ptr(), n_payload + 2, n_payload + 2, Cn, ref.data_ptr(), nref, s)
    cnt = torch.zeros((Cn, 2), dtype=torch.int32, device="cuda")
    check = (0, 4097, lo + 5, Cn - 1)
    ods = {c: orc.QPSKDeModulator(fs, rs, **kw) for c in check}
    for burst in range(4):
        ch.apply_dev(tx.data_ptr(), ff, ff, rxs.data_ptr(), ff, s)
        dem.demod_bits_dev(rxs.data_ptr(), ff, ff, bits.data_ptr(), cap, nb.data_ptr(), s)
        gpu.ber_count_dev(bits.data_ptr(), cap, nb.data_ptr(), ref.data_ptr(), nref, nref, Cn, cnt.data_ptr(), s)
        block = rxs[lo:hi].contiguous()
        sub.demod_bits_dev(block.data_ptr(), ff, ff, sbits.data_ptr(), cap, snb.data_ptr(), s)
        torch.cuda.synchronize()
        nb_h = nb.cpu().numpy()
        assert torch.equal(snb, nb[lo:hi]), burst                          # (ii)
        for k in range(hi - lo):
            assert torch.equal(sbits[k, : nb_h[lo + k]], bits[lo + k, : nb_h[lo + k]]), (burst, lo + k)
        for c, od in ods.items():                                          # (i)
            want = od.DeModulate(rxs[c].cpu().numpy())
            got = "".join("1" if b else "0" for b in bits[c, : nb_h[c]].cpu().numpy())
            assert got == want, (burst, c)
    # (iii) the counters of the last burst against a recount on the host (bits past the reference count as errors)
    cnt_h, bits_h, ref_h = cnt.cpu().numpy(), bits.cpu().numpy(), ref.cpu().numpy()
    for c in list(range(0, Cn, 1021)) + [Cn - 1]:
        n = min(int(nb_h[c]), nref)
        err = int((bits_h[c, :n] != ref_h[c, :n]).sum()) + (nref - n)
        assert cnt_h[c].tolist() == [err, nref], c
    locked = float((cnt_h[:, 0] == 0).mean())
    print(f"config4 use_fll={use_fll}: error-free channels in burst 4: {locked:.3f}")
    assert locked > (0.2 if use_fll else 0.5), locked                     # (iv) measured 0.67 / 0.51: the rest lose a burst exactly as the reference does


# ---- SURVEY §8f-4: packed-bit I/O ------------------------------------------------------------------
@pytest.mark.parametrize("tlen", [1, 3, 8, 31, 32, 33, 63, 64, 65, 100])
def test_demod_tsc_strip_lengths(gpu, orc, tlen):
    """TSC strip (QPSKDeModulator.cs:413-422): the bit-parallel search serves 1..64-bit sequences, longer ones take the
    byte search; both must cut where the oracle's IndexOf does (or return "" when the sequence is absent)."""
    rng = np.random.default_rng(100 + tlen)
    tsc = "".join(rng.choice(["0", "1"], tlen))
    fs, rs = 4000, 1000
    mod = orc.QPSKModulator(fs, rs, 0.35, 10, True, tsc)
    x = np.concatenate([mod.Modulate(_bits(2 * (150 + 7 * k), 7 + k)) for k in range(3)])
    kw = dict(RrcAlpha=0.35, rrcSpan=10, SymbolSyncBandwith=0.002, tsc=tsc)
    want = orc.QPSKDeModulator(fs, rs, **kw).DeModulate(x)
    got = gpu.QPSKDeModulator(fs, rs, **kw).DeModulate(x)
    assert got == want
    # a sequence that is not in the stream, and one with a character that is neither '0' nor '1'
    for absent in ("01" * 30 + "0011", tsc[:-1] + "x" if tlen > 1 else "x"):
        kw2 = dict(kw, tsc=absent)
        assert gpu.QPSKDeModulator(fs, rs, **kw2).DeModulate(x) == orc.QPSKDeModulator(fs, rs, **kw2).DeModulate(x)


def _tsc_smem_bytes(L, T, sps):
    """Shared memory DemodEngine::bits_dev asks for tsc_strip_smem_kernel on an L-sample call (rows of 2 x the symbol
    bound, padded to 16 bytes); above 160 KB the call takes tsc_strip_kernel."""
    sl = L if sps - 0.1 <= 1.0 else min(int((L + 4) / (sps - 0.1)) + 2, L)
    ld_raw = (2 * max(sl, 1) + 15) & ~15
    row_bytes = (ld_raw + 15) & ~15
    words = (row_bytes + 31) // 32 + 4
    return 4 * (row_bytes + ((T + 15) & ~15)) + 16 * words


@pytest.mark.parametrize("C", [1, 33])
@pytest.mark.parametrize("tlen", [64, 100])
def test_demod_tsc_strip_long_calls(gpu, orc, tlen, C):
    """Calls too long for tsc_strip_smem_kernel's shared memory take tsc_strip_kernel: three calls per channel, the first
    with the TSC in its middle, the second without it and ending half-way through the next TSC, which the third call
    starts in.  Bits must equal the oracle's on every call."""
    import re
    import symsync_dispatch as sd
    fs, rs, span = 2000, 1000, 10
    sps = fs / rs
    tsc = "".join(np.random.default_rng(200 + tlen).choice(["0", "1"], tlen))
    Lmin = next(L for L in range(20000, 60000, 16) if _tsc_smem_bytes(L, tlen, sps) > 160 * 1024)
    n_bits = 2 * ((Lmin + 1200) // 2)                            # ~ one sample per bit at sps 2
    # the TSC goes inside a frame's bit string: at the start of a frame the differential reference of the modulator
    # restarts while the demodulator's carries on, and the first dibit would not decode as sent
    mod = orc.QPSKModulator(fs, rs, 0.35, span, True, None)
    lead = 1000                                                  # bits of t before its TSC
    rows, cuts = [], None
    for c in range(C):
        a = mod.Modulate(_bits(n_bits // 2, 3 * c) + tsc + _bits(n_bits // 2, 3 * c + 1))
        b = mod.Modulate(_bits(n_bits, 3 * c + 2))
        t = mod.Modulate(_bits(lead, 3 * c + 3) + tsc + _bits(n_bits, 3 * c + 4))
        rng = np.random.default_rng(c)
        z = np.concatenate([a, b, t])
        rows.append((z + 0.01 * rng.standard_normal(z.size)).astype(np.float32))
        mid = lead + span * int(sps) // 2 + tlen // 2            # about the middle of t's TSC, in samples
        cuts = [0, a.size // 2, a.size // 2 + b.size // 2 + mid, z.size // 2]
    x = np.stack(rows)
    assert min(q - p for p, q in zip(cuts[:-1], cuts[1:])) >= Lmin
    kw = dict(RrcAlpha=0.35, rrcSpan=span, SymbolSyncBandwith=0.002, tsc=tsc)
    gd = gpu.QPSKDeModulator(fs, rs, channels=C, **kw)
    ods = [orc.QPSKDeModulator(fs, rs, **kw) for _ in range(C)]
    for k, (p, q) in enumerate(zip(cuts[:-1], cuts[1:])):
        xs = np.ascontiguousarray(x[:, 2 * p:2 * q])
        arg = xs if C > 1 else xs[0]
        if k == 0:
            got, names = sd.launched_kernels(lambda: gd.DeModulate(arg))
            print(f"[kernel] tsc long call T={tlen} C={C}: {sorted(set(n.split('(')[0] for n in names if 'tsc_strip' in n))}")
            assert any(re.search(r"\btsc_strip_kernel\b", n) for n in names), names
            assert not any("tsc_strip_smem_kernel" in n for n in names), names
        else:
            got = gd.DeModulate(arg)
        got = got if C > 1 else [got]
        for c in range(C):
            want = ods[c].DeModulate(xs[c])
            assert got[c] == want, (k, c)
            assert (want != "") == (k == 0), (k, c, len(want))    # found in the first call only: absent, then cut in two


@pytest.mark.parametrize("diff,tsc,nbits", [(True, TSC, 600), (False, None, 4096), (True, None, 13), (True, TSC, 0), (False, TSC, 7)])
def test_modulate_packed_equals_bit_string(gpu, orc, diff, tsc, nbits):
    rng = np.random.default_rng(nbits + 1)
    packed = bytes(rng.integers(0, 256, (nbits + 7) // 8, dtype=np.uint8))
    bits = orc.BitPacker.BytesToBitString(packed)[:nbits]
    fs = 8_000_000
    want = orc.QPSKModulator(fs, fs // 4, 0.35, 8, diff, tsc).Modulate(bits)
    m = gpu.QPSKModulator(fs, fs // 4, 0.35, 8, diff, tsc)
    got = m.ModulatePacked(packed, nbits)
    assert got.shape == want.shape
    assert np.array_equal(got, m.Modulate(bits))                     # bit-identical to the char-string form
    if want.size:
        assert np.abs(got - want).max() <= 1e-5 * np.abs(want).max()
    with pytest.raises(gpu.ArgumentException):
        m.ModulatePacked(packed, 8 * len(packed) + 1)


@pytest.mark.parametrize("tsc", [None, TSC])
def test_demodulate_packed_equals_bit_string(gpu, orc, tsc):
    fs = 10_000_000
    a = float(np.float32(0.4))
    tx = orc.QPSKModulator(fs, fs // 2, a, 10, tsc=tsc).Modulate(_bits(1003 * 2, 41))
    d1 = gpu.QPSKDeModulator(fs, fs // 2, a, 10, tsc=tsc)
    d2 = gpu.QPSKDeModulator(fs, fs // 2, a, 10, tsc=tsc)
    od = orc.QPSKDeModulator(fs, fs // 2, a, 10, tsc=tsc)
    for _ in range(3):                                               # state carried; odd and even bit counts
        bits = d1.DeModulate(tx)
        packed, nb = d2.DeModulatePacked(tx)
        assert nb == len(bits)
        assert bits == od.DeModulate(tx)
        full = orc.BitPacker.BitsToBytes(bits, 0)                    # drops the trailing incomplete byte
        assert packed[: len(full)] == full
        if nb % 8:
            tail = bits[8 * len(full):]
            assert packed[len(full)] == int(tail.ljust(8, "0"), 2)
        assert len(packed) == (nb + 7) // 8
    # batch handle: every channel equals the single-stream result
    C = 3
    xs = np.stack([orc.QPSKModulator(fs, fs // 2, a, 10, tsc=tsc).Modulate(_bits(800 + 2 * c, 50 + c))[: 2 * 800] for c in range(C)])
    db = gpu.QPSKDeModulator(fs, fs // 2, a, 10, tsc=tsc, channels=C)
    outs = db.DeModulatePacked(xs)
    for c in range(C):
        one = gpu.QPSKDeModulator(fs, fs // 2, a, 10, tsc=tsc).DeModulatePacked(xs[c])
        assert outs[c] == one


def test_pack_bits_dev_ragged(gpu):
    import torch
    rng = np.random.default_rng(3)
    C, ld = 6, 1032
    bits = rng.integers(0, 2, (C, ld), dtype=np.uint8)
    nb = np.array([0, 1, 7, 8, 1001, 1032], np.int64)
    db, dn = torch.from_numpy(bits).cuda(), torch.from_numpy(nb).cuda()
    out = torch.full((C, ld // 8), 0xEE, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    gpu.pack_bits_dev(db.data_ptr(), ld, dn.data_ptr(), ld, C, out.data_ptr(), ld // 8)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    for c in range(C):
        n = int(nb[c])
        want = np.packbits(bits[c, :n])                               # MSB first, zero-padded tail
        assert np.array_equal(got[c, : want.size], want)
        assert (got[c, want.size:] == 0xEE).all()                     # nothing written past the last used byte
